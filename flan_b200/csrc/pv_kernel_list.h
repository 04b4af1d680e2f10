// flan_b200/csrc/pv_kernel_list.h -- the transform kernels a release build carries: exactly those the launch policy
// (pv_policy.h: choose_analysis / choose_synthesis) can return. pv_kernels.cu instantiates them from this list and the
// emulator enumerates it. X-macro: PV_RELEASE_KERNELS( A, AM, S, SM ) expands
//   A( N, PT, TPS, ONE, PAD, EMIT )    pv_analysis_kernel
//   AM( N, TPS )                       pv_analysis_mirror_kernel
//   S( N, TPS, ONE )                   pv_synthesis_kernel
//   SM( N, TPS, ONE, GEN )             pv_synthesis_mirror_kernel
#pragma once

#define PV_RELEASE_KERNELS( A, AM, S, SM )                                                                         \
	A( 256, 8, 768, false, false, false )                                                                           \
	A( 512, 8, 768, false, false, false )                                                                           \
	A( 1024, 8, 768, false, false, false )                                                                          \
	A( 2048, 8, 768, false, false, false )                                                                          \
	A( 2048, 16, 512, true, false, false ) A( 2048, 16, 512, true, true, false ) A( 2048, 16, 512, true, false, true ) \
	A( 4096, 16, 512, true, false, false ) A( 4096, 16, 512, true, true, false ) A( 4096, 16, 512, true, false, true ) \
	A( 8192, 16, 512, true, false, false ) A( 8192, 16, 512, true, true, false ) A( 8192, 16, 512, true, false, true ) \
	AM( 1024, 512 )                                                                                                 \
	S( 256, 768, false ) S( 512, 768, false ) S( 1024, 768, false ) S( 2048, 768, false ) S( 4096, 768, false )     \
	S( 8192, 1024, true )                                                                                           \
	SM( 1024, 384, false, false ) SM( 1024, 384, false, true )                                                      \
	SM( 2048, 384, false, false ) SM( 2048, 384, false, true )                                                      \
	SM( 4096, 512, true, false ) SM( 4096, 384, false, true )                                                       \
	SM( 8192, 512, true, false ) SM( 8192, 512, true, true )
