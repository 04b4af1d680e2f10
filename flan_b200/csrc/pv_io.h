// flan_b200/csrc/pv_io.h -- launch interface of pv_io.cu: sample codecs of the file formats either side of the path
// (.flan RIFF-PV, PV/PVBuffer.cpp:99-140,216-273; WAV through libsndfile, Audio/AudioBuffer.cpp:80-192).
#pragma once

#include <cuda_runtime.h>
#include <cstdint>

namespace pvio {

// count = MF elements; bytes = 6 * count, 16-byte aligned.
cudaError_t launch_flan_encode( const float * pv, int64_t count, float dft_size, float sample_rate, uint8_t * bytes, int sms, cudaStream_t st );
cudaError_t launch_flan_decode( const uint8_t * bytes, int64_t count, float dft_size, float sample_rate, float * pv, int sms, cudaStream_t st );

// Bytes a value of a WAV sample type (FLAN_B200_WAV_*) takes; 0 for a code that is not one.
int pcm_width( int subtype );
// audio: n frames of planar float[C][stride]; bytes: interleaved frames, pcm_width( subtype ) * C * n, 16-byte aligned.
// An unknown subtype launches nothing and returns cudaErrorInvalidValue.
cudaError_t launch_pcm_encode( int subtype, const float * audio, int C, int64_t stride, int64_t n, uint8_t * bytes, int sms, cudaStream_t st );
cudaError_t launch_pcm_decode( int subtype, const uint8_t * bytes, int C, int64_t stride, int64_t n, float * audio, int sms, cudaStream_t st );

} // namespace pvio
