// flan_b200/csrc/pv_capi_io.cu -- C ABI of the file formats either side of the path (SURVEY 8f-4): .flan RIFF-PV
// (PV/PVBuffer.cpp:99-140,216-273) and WAV with libsndfile's sample types for it (Audio/AudioBuffer.cpp:80-192). Headers on
// the host, sample codecs on the device (pv_io.cu), streamed in chunks through a pinned buffer.
#include "pv_ctx.h"

#include <cstdio>
#include <cstdlib>

using namespace pvrt;

// ---- file formats either side of the path (SURVEY 8f-4) ------------------------------------------

namespace {

void put16( std::vector<uint8_t> & b, uint16_t v ) { b.push_back( v & 0xFF ); b.push_back( v >> 8 ); }
void put32( std::vector<uint8_t> & b, uint32_t v ) { for( int i = 0; i < 4; ++i ) b.push_back( ( v >> ( 8 * i ) ) & 0xFF ); }
void put4c( std::vector<uint8_t> & b, const char * s ) { for( int i = 0; i < 4; ++i ) b.push_back( (uint8_t)( *s ? *s++ : 0 ) ); }
uint16_t get16( const uint8_t * p ) { return (uint16_t)( p[0] | ( p[1] << 8 ) ); }
uint32_t get32( const uint8_t * p ) { return (uint32_t) p[0] | ( (uint32_t) p[1] << 8 ) | ( (uint32_t) p[2] << 16 ) | ( (uint32_t) p[3] << 24 ); }

struct FileCloser { FILE * f; ~FileCloser() { if( f ) std::fclose( f ); } };
struct PinnedBuf { void * p = nullptr; ~PinnedBuf() { if( p ) cudaFreeHost( p ); } };

constexpr int64_t IO_CHUNK_BYTES = int64_t( 192 ) << 20;        // file bytes per staging chunk

// Streams `values` samples of `width` bytes between a file and the device in chunks of at most `max_chunk` values through
// ctx scratch + a pinned buffer. launch( first_value, n_values, d_bytes ) runs the codec for one chunk.
template<class Launch> int stream_file( flan_b200_ctx * ctx, FILE * f, bool writing, int64_t values, int width, int64_t max_chunk, Launch launch )
	{
	const int64_t chunk = values < max_chunk ? ( values > 0 ? values : 1 ) : max_chunk;
	const size_t chunk_bytes = (size_t) chunk * width;
	void * ws = nullptr;
	int rc = get_workspace( ctx, chunk_bytes + 16, &ws );
	if( rc ) return rc;
	PinnedBuf host;
	CK( cudaMallocHost( &host.p, chunk_bytes ), "pinned staging buffer" );
	for( int64_t v0 = 0; v0 < values; v0 += chunk )
		{
		const int64_t nv = values - v0 < chunk ? values - v0 : chunk;
		const size_t nb = (size_t) nv * width;
		if( writing )
			{
			CK( launch( v0, nv, (uint8_t *) ws ), "codec launch" );
			CK( cudaMemcpyAsync( host.p, ws, nb, cudaMemcpyDeviceToHost, ctx->compute ), "download" );
			CK( cudaStreamSynchronize( ctx->compute ), "download sync" );
			if( std::fwrite( host.p, 1, nb, f ) != nb ) return fail( ctx, FLAN_B200_INVALID, "short write" );
			}
		else
			{
			if( std::fread( host.p, 1, nb, f ) != nb ) return fail( ctx, FLAN_B200_INVALID, "file is shorter than its header says" );
			CK( cudaMemcpyAsync( ws, host.p, nb, cudaMemcpyHostToDevice, ctx->compute ), "upload" );
			CK( launch( v0, nv, (uint8_t *) ws ), "codec launch" );
			CK( cudaStreamSynchronize( ctx->compute ), "upload sync" );
			}
		ctx->launches++;
		}
	return FLAN_B200_OK;
	}

// .flan values (three bytes each) per staging chunk: 2^26, a multiple of 4096.
constexpr int64_t FLAN_CHUNK_VALUES = IO_CHUNK_BYTES / 3;

// Frames of interleaved samples per staging chunk: about IO_CHUNK_BYTES of file, a multiple of 4096 frames (so a chunk
// starts 16-byte aligned at every width), never zero however many channels the (untrusted, 16-bit) header field claims.
int64_t wav_frames_per_chunk( int C, int width )
	{
	const int64_t f = ( IO_CHUNK_BYTES / width / ( C > 0 ? C : 1 ) ) / 4096 * 4096;
	return f > 0 ? f : 4096;
	}

struct FlanHeader { int C = 0; int64_t F = 0; int B = 0; uint32_t sr = 0, hop = 0, window = 0; long data_offset = 0; };

// Reads the chunks the way PVBuffer::load does (PVBuffer.cpp:231-250): fixed order RIFF / fmt / data.
int read_flan_header( flan_b200_ctx * ctx, FILE * f, FlanHeader & h )
	{
	uint8_t b[58];
	if( std::fread( b, 1, 58, f ) != 58 ) return fail( ctx, FLAN_B200_INVALID, "not a PV file: too short" );
	if( std::memcmp( b, "RIFF", 4 ) != 0 ) return fail( ctx, FLAN_B200_INVALID, "isn't a correctly formatted RIFF file" );
	if( std::strncmp( (const char *) b + 8, "PV", 4 ) != 0 ) return fail( ctx, FLAN_B200_INVALID, "isn't a PV file" );
	if( std::memcmp( b + 12, "fmt ", 4 ) != 0 ) return fail( ctx, FLAN_B200_INVALID, "\"fmt \" wasn't at the start of the format chunk" );
	if( get16( b + 20 ) != 1 ) return fail( ctx, FLAN_B200_INVALID, "Formatting must be 1 (signed int)." );
	h.C = get16( b + 22 ); h.F = get32( b + 24 );
	const uint32_t bins = get32( b + 28 );
	// the fields come from a file: a dft size of (B-1)*2 needs B >= 2, and C*F*B must stay far inside int64
	if( h.C < 1 || bins < 2 || bins > ( 1u << 30 ) ) return fail( ctx, FLAN_B200_INVALID, "PV file header has no channels or an impossible bin count" );
	h.B = (int) bins;
	h.sr = get32( b + 32 ); h.hop = get32( b + 36 ); h.window = get32( b + 40 );
	if( get32( b + 44 ) != 24 ) return fail( ctx, FLAN_B200_INVALID, "Bit depth must be 24." );
	if( get16( b + 48 ) != 1 ) return fail( ctx, FLAN_B200_INVALID, "PV window must be 1 (hann)." );
	if( std::memcmp( b + 50, "data", 4 ) != 0 ) return fail( ctx, FLAN_B200_INVALID, "\"data\" wasn't at the start of the data chunk" );
	h.data_offset = 58;
	return FLAN_B200_OK;
	}

struct WavHeader { int C = 0; int64_t n = 0; uint32_t sr = 0; int subtype = 0; long data_offset = 0; };

// The FLAN_B200_WAV_* type of a fmt chunk's fields, or 0. width = block_align / channels, the container.
int wav_subtype( int tag, int bits, int width )
	{
	if( tag == 1 && bits >= 1 && bits <= 32 && width == ( bits + 7 ) / 8 )
		{
		const int by_width[5] = { 0, FLAN_B200_WAV_PCM_U8, FLAN_B200_WAV_PCM_16, FLAN_B200_WAV_PCM_24, FLAN_B200_WAV_PCM_32 };
		return by_width[width];
		}
	if( tag == 3 && bits == 32 && width == 4 ) return FLAN_B200_WAV_FLOAT;
	if( tag == 3 && bits == 64 && width == 8 ) return FLAN_B200_WAV_DOUBLE;
	return 0;
	}

int read_wav_header( flan_b200_ctx * ctx, FILE * f, WavHeader & h )
	{
	uint8_t b[12];
	if( std::fread( b, 1, 12, f ) != 12 || std::memcmp( b, "RIFF", 4 ) != 0 || std::memcmp( b + 8, "WAVE", 4 ) != 0 )
		return fail( ctx, FLAN_B200_INVALID, "not a RIFF/WAVE file" );
	bool have_fmt = false;
	int bits = 0, tag = 0, block = 0;
	for( ;; )
		{
		uint8_t c[8];
		if( std::fread( c, 1, 8, f ) != 8 ) return fail( ctx, FLAN_B200_INVALID, "WAVE file without a data chunk" );
		const uint32_t size = get32( c + 4 );
		if( std::memcmp( c, "fmt ", 4 ) == 0 )
			{
			uint8_t m[40] = { 0 };
			const uint32_t take = size < 40 ? size : 40;
			if( size < 16 || std::fread( m, 1, take, f ) != take ) return fail( ctx, FLAN_B200_INVALID, "bad fmt chunk" );
			tag = get16( m ); h.C = get16( m + 2 ); h.sr = get32( m + 4 ); block = get16( m + 12 ); bits = get16( m + 14 );
			if( tag == 0xFFFE && size >= 40 )               // WAVE_FORMAT_EXTENSIBLE: the sub-format GUID's tail is the
				{                                           // one KSDATAFORMAT_SUBTYPE_PCM / _IEEE_FLOAT share
				static const uint8_t tail[14] = { 0x00, 0x00, 0x00, 0x00, 0x10, 0x00, 0x80, 0x00, 0x00, 0xAA, 0x00, 0x38, 0x9B, 0x71 };
				if( std::memcmp( m + 26, tail, 14 ) == 0 ) tag = get16( m + 24 );
				}
			std::fseek( f, (long)( size - take + ( size & 1 ) ), SEEK_CUR );
			have_fmt = true;
			}
		else if( std::memcmp( c, "data", 4 ) == 0 )
			{
			if( !have_fmt ) return fail( ctx, FLAN_B200_INVALID, "data chunk before fmt chunk" );
			const int width = h.C > 0 ? block / h.C : 0;
			h.subtype = ( h.C > 0 && block == width * h.C ) ? wav_subtype( tag, bits, width ) : 0;
			if( !h.subtype )
				return fail( ctx, FLAN_B200_UNSUPPORTED, "WAVE format tag " + std::to_string( tag ) + " with " + std::to_string( bits ) +
				             " bits, block align " + std::to_string( block ) + " for " + std::to_string( h.C ) +
				             " channels: only PCM (8, 16, 24, 32 bits) and IEEE float (32, 64 bits) samples are decoded on the device" );
			h.n = (int64_t) size / block;
			h.data_offset = std::ftell( f );
			return FLAN_B200_OK;
			}
		else std::fseek( f, (long)( size + ( size & 1 ) ), SEEK_CUR );
		}
	}

int check_subtype( flan_b200_ctx * ctx, int subtype )
	{
	return pvio::pcm_width( subtype ) ? FLAN_B200_OK : fail( ctx, FLAN_B200_INVALID, "unknown WAV sample type " + std::to_string( subtype ) );
	}

} // namespace

extern "C" {

int flan_b200_flan_encode( flan_b200_ctx * ctx, const float * d_pv, int64_t count, float dft_size, float sr, uint8_t * d_bytes )
	{
	if( !ctx || count < 0 || ( count && ( !d_pv || !d_bytes ) ) ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_pv, d_bytes } );
	if( count == 0 ) return FLAN_B200_OK;
	{ LaunchTimer lt( ctx, 8 ); CK( pvio::launch_flan_encode( d_pv, count, dft_size, sr, d_bytes, ctx->sms, ctx->compute ), "flan encode launch" ); }
	return FLAN_B200_OK;
	}

int flan_b200_flan_decode( flan_b200_ctx * ctx, const uint8_t * d_bytes, int64_t count, float dft_size, float sr, float * d_pv )
	{
	if( !ctx || count < 0 || ( count && ( !d_pv || !d_bytes ) ) ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_bytes, d_pv } );
	if( count == 0 ) return FLAN_B200_OK;
	ctx->summaries.drop();          // new rows, written without the workspace
	{ LaunchTimer lt( ctx, 8 ); CK( pvio::launch_flan_decode( d_bytes, count, dft_size, sr, d_pv, ctx->sms, ctx->compute ), "flan decode launch" ); }
	return FLAN_B200_OK;
	}

int flan_b200_pcm_encode( flan_b200_ctx * ctx, const float * d_audio, int C, int64_t n, int subtype, uint8_t * d_bytes )
	{
	if( !ctx || C < 1 || n < 0 || ( n && ( !d_audio || !d_bytes ) ) ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	if( int rc = check_subtype( ctx, subtype ) ) return rc;
	BlockUse use( ctx, { d_audio, d_bytes } );
	if( n == 0 ) return FLAN_B200_OK;
	{ LaunchTimer lt( ctx, 8 ); CK( pvio::launch_pcm_encode( subtype, d_audio, C, n, n, d_bytes, ctx->sms, ctx->compute ), "pcm encode launch" ); }
	return FLAN_B200_OK;
	}

int flan_b200_pcm_decode( flan_b200_ctx * ctx, const uint8_t * d_bytes, int C, int64_t n, int subtype, float * d_audio )
	{
	if( !ctx || C < 1 || n < 0 || ( n && ( !d_audio || !d_bytes ) ) ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	if( int rc = check_subtype( ctx, subtype ) ) return rc;
	BlockUse use( ctx, { d_bytes, d_audio } );
	if( n == 0 ) return FLAN_B200_OK;
	{ LaunchTimer lt( ctx, 8 ); CK( pvio::launch_pcm_decode( subtype, d_bytes, C, n, n, d_audio, ctx->sms, ctx->compute ), "pcm decode launch" ); }
	return FLAN_B200_OK;
	}

int flan_b200_pcm24_encode( flan_b200_ctx * ctx, const float * d_audio, int C, int64_t n, uint8_t * d_bytes )
	{
	return flan_b200_pcm_encode( ctx, d_audio, C, n, FLAN_B200_WAV_PCM_24, d_bytes );
	}

int flan_b200_pcm24_decode( flan_b200_ctx * ctx, const uint8_t * d_bytes, int C, int64_t n, float * d_audio )
	{
	return flan_b200_pcm_decode( ctx, d_bytes, C, n, FLAN_B200_WAV_PCM_24, d_audio );
	}

int flan_b200_save_flan( flan_b200_ctx * ctx, const char * path, const float * d_pv, int C, int64_t F, int B,
                         float sr, float ar, int window_size )
	{
	if( !ctx || !path || C < 0 || F < 0 || B < 0 ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_pv } );
	const int64_t count = (int64_t) C * F * B;
	if( count && !d_pv ) return FLAN_B200_INVALID;
	FileCloser file{ std::fopen( path, "wb" ) };
	if( !file.f ) return fail( ctx, FLAN_B200_INVALID, std::string( "Error opening " ) + path + " to write RIFF." );
	std::vector<uint8_t> h;                                              // Utility/Bytes.cpp:70-112, PVBuffer.cpp:128-139
	put4c( h, "RIFF" ); put32( h, 4 ); put4c( h, "PV" );
	put4c( h, "fmt " ); put32( h, 30 );
	put16( h, 1 ); put16( h, (uint16_t) C ); put32( h, (uint32_t) F ); put32( h, (uint32_t) B );
	put32( h, (uint32_t) sr ); put32( h, (uint32_t) flan_b200_hop_from_rates( sr, ar ) ); put32( h, (uint32_t) window_size );
	put32( h, 24 ); put16( h, 1 );
	put4c( h, "data" ); put32( h, (uint32_t)( count * 6 ) );
	if( std::fwrite( h.data(), 1, h.size(), file.f ) != h.size() ) return fail( ctx, FLAN_B200_INVALID, "short write" );
	const float dft = float( ( B - 1 ) * 2 );                            // window_size_f = get_dft_size(), PVBuffer.cpp:103
	return stream_file( ctx, file.f, true, 2 * count, 3, FLAN_CHUNK_VALUES, [&]( int64_t v0, int64_t nv, uint8_t * d_bytes )
		{ return pvio::launch_flan_encode( d_pv + v0, nv / 2, dft, sr, d_bytes, ctx->sms, ctx->compute ); } );
	}

int flan_b200_flan_info( flan_b200_ctx * ctx, const char * path, int * C, int64_t * F, int * B, float * sr, float * rate_field, int * window_size )
	{
	if( !ctx || !path ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	FileCloser file{ std::fopen( path, "rb" ) };
	if( !file.f ) return fail( ctx, FLAN_B200_INVALID, std::string( "Error opening " ) + path + " to load PV." );
	FlanHeader h;
	int rc = read_flan_header( ctx, file.f, h );
	if( rc ) return rc;
	if( C ) *C = h.C; if( F ) *F = h.F; if( B ) *B = h.B;
	if( sr ) *sr = float( h.sr ); if( rate_field ) *rate_field = float( h.hop ); if( window_size ) *window_size = (int) h.window;
	return FLAN_B200_OK;
	}

int flan_b200_load_flan( flan_b200_ctx * ctx, const char * path, float * d_pv, int64_t capacity )
	{
	if( !ctx || !path ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_pv } );
	FileCloser file{ std::fopen( path, "rb" ) };
	if( !file.f ) return fail( ctx, FLAN_B200_INVALID, std::string( "Error opening " ) + path + " to load PV." );
	FlanHeader h;
	int rc = read_flan_header( ctx, file.f, h );
	if( rc ) return rc;
	if( (long double) h.C * (long double) h.F * (long double) h.B > (long double) capacity )      // the product itself may not fit int64
		return fail( ctx, FLAN_B200_INVALID, "destination holds fewer MF elements than the file" );
	const int64_t count = (int64_t) h.C * h.F * h.B;
	if( count > capacity || ( count && !d_pv ) ) return fail( ctx, FLAN_B200_INVALID, "destination holds fewer MF elements than the file" );
	const float dft = float( ( h.B - 1 ) * 2 ), sr = float( h.sr );
	return stream_file( ctx, file.f, false, 2 * count, 3, FLAN_CHUNK_VALUES, [&]( int64_t v0, int64_t nv, uint8_t * d_bytes )
		{ return pvio::launch_flan_decode( d_bytes, nv / 2, dft, sr, d_pv + v0, ctx->sms, ctx->compute ); } );
	}

int flan_b200_save_wav_as( flan_b200_ctx * ctx, const char * path, const float * d_audio, int C, int64_t n, float sr, int subtype )
	{
	if( !ctx || !path || C < 1 || n < 0 || ( n && !d_audio ) ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	if( int rc = check_subtype( ctx, subtype ) ) return rc;
	BlockUse use( ctx, { d_audio } );
	const int width = pvio::pcm_width( subtype );
	const bool ieee = subtype == FLAN_B200_WAV_FLOAT || subtype == FLAN_B200_WAV_DOUBLE;
	// PCM: RIFF, fmt (16), data = 44 bytes. Float: RIFF, fmt (18, cbSize 0), fact (frame count), data = 58 bytes.
	const int64_t header = ieee ? 58 : 44;
	const int64_t room = 0xFFFFFFFFll - ( header - 8 );                   // largest data chunk, pad byte included
	if( n > room / ( (int64_t) C * width ) || (int64_t) C * n * width + ( ( (int64_t) C * n * width ) & 1 ) > room )
		return fail( ctx, FLAN_B200_UNSUPPORTED, "signal exceeds the 4 GiB RIFF limit" );
	FileCloser file{ std::fopen( path, "wb" ) };
	if( !file.f ) return fail( ctx, FLAN_B200_INVALID, std::string( path ) + " could not be opened for saving." );
	const uint32_t data_bytes = (uint32_t)( (int64_t) C * n * width );
	std::vector<uint8_t> h;
	put4c( h, "RIFF" ); put32( h, (uint32_t)( header - 8 ) + data_bytes + ( data_bytes & 1 ) ); put4c( h, "WAVE" );
	put4c( h, "fmt " ); put32( h, ieee ? 18 : 16 ); put16( h, ieee ? 3 : 1 ); put16( h, (uint16_t) C ); put32( h, (uint32_t) sr );
	put32( h, (uint32_t) sr * width * C ); put16( h, (uint16_t)( width * C ) ); put16( h, (uint16_t)( 8 * width ) );
	if( ieee ) { put16( h, 0 ); put4c( h, "fact" ); put32( h, 4 ); put32( h, (uint32_t) n ); }
	put4c( h, "data" ); put32( h, data_bytes );
	if( std::fwrite( h.data(), 1, h.size(), file.f ) != h.size() ) return fail( ctx, FLAN_B200_INVALID, "short write" );
	// the interleaved order makes a chunk of values a range of FRAMES of the planar buffer
	const int64_t frames_per_chunk = wav_frames_per_chunk( C, width );
	int rc = stream_file( ctx, file.f, true, (int64_t) C * n, width, frames_per_chunk * C, [&]( int64_t v0, int64_t nv, uint8_t * d_bytes )
		{ return pvio::launch_pcm_encode( subtype, d_audio + v0 / C, C, n, nv / C, d_bytes, ctx->sms, ctx->compute ); } );
	if( rc ) return rc;
	if( data_bytes & 1 ) { const uint8_t pad = 0; std::fwrite( &pad, 1, 1, file.f ); }
	return FLAN_B200_OK;
	}

int flan_b200_save_wav( flan_b200_ctx * ctx, const char * path, const float * d_audio, int C, int64_t n, float sr )
	{
	return flan_b200_save_wav_as( ctx, path, d_audio, C, n, sr, FLAN_B200_WAV_PCM_24 );
	}

static int open_wav( flan_b200_ctx * ctx, const char * path, FileCloser & file, WavHeader & h )
	{
	file.f = std::fopen( path, "rb" );
	if( !file.f ) return fail( ctx, FLAN_B200_INVALID, std::string( path ) + " could not be opened." );
	return read_wav_header( ctx, file.f, h );
	}

int flan_b200_wav_info( flan_b200_ctx * ctx, const char * path, int * C, int64_t * n, float * sr )
	{
	if( !ctx || !path ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	FileCloser file{ nullptr };
	WavHeader h;
	if( int rc = open_wav( ctx, path, file, h ) ) return rc;
	if( C ) *C = h.C; if( n ) *n = h.n; if( sr ) *sr = float( h.sr );
	return FLAN_B200_OK;
	}

int flan_b200_wav_format( flan_b200_ctx * ctx, const char * path, int * subtype )
	{
	if( !ctx || !path ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	FileCloser file{ nullptr };
	WavHeader h;
	if( int rc = open_wav( ctx, path, file, h ) ) return rc;
	if( subtype ) *subtype = h.subtype;
	return FLAN_B200_OK;
	}

int flan_b200_load_wav( flan_b200_ctx * ctx, const char * path, float * d_audio, int64_t capacity )
	{
	if( !ctx || !path ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_audio } );
	FileCloser file{ nullptr };
	WavHeader h;
	if( int rc = open_wav( ctx, path, file, h ) ) return rc;
	const int64_t values = (int64_t) h.C * h.n;
	if( values > capacity || ( values && !d_audio ) ) return fail( ctx, FLAN_B200_INVALID, "destination holds fewer samples than the file" );
	std::fseek( file.f, h.data_offset, SEEK_SET );
	const int width = pvio::pcm_width( h.subtype );
	const int64_t frames_per_chunk = wav_frames_per_chunk( h.C, width );
	return stream_file( ctx, file.f, false, values, width, frames_per_chunk * h.C, [&]( int64_t v0, int64_t nv, uint8_t * d_bytes )
		{ return pvio::launch_pcm_decode( h.subtype, d_bytes, h.C, h.n, nv / h.C, d_audio + v0 / h.C, ctx->sms, ctx->compute ); } );
	}

} // extern "C"
