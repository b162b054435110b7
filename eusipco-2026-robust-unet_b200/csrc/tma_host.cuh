// Host-side CUtensorMap construction (cuTensorMapEncodeTiled through the runtime's driver entry point,
// so the library has no link-time dependency on libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rbunet.h"

// Encode a bf16 tensor map with SWIZZLE_128B. dims/strides innermost first; strides[i] is the byte stride
// of dimension i+1 (dimension 0 is contiguous). Returns 0 on success (error text via rbu_set_error).
int rbu_encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                         const uint64_t* strides_bytes, const uint32_t* box);
// Same with SWIZZLE_64B (swizzle_bytes == 64; inner box extent <= 64 bytes) or SWIZZLE_128B (128).
int rbu_encode_tmap_bf16_sw(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                            const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes);

// conv_halo.cu: halo-reuse variant of the implicit-GEMM convolution (3x3 dilation 1 / 1x1 segments).
int rbu_conv_halo_supported(const rbu_conv_gemm_args* a);
int rbu_conv_halo_launch(const rbu_conv_gemm_args* a, cudaStream_t stream);

// wgrad_halo.cu: all-taps-from-one-halo variant of the weight-gradient GEMM (3x3, dilation 1).
int rbu_wgrad_halo_supported(const rbu_wgrad_args* a);
size_t rbu_wgrad_halo_workspace_bytes(const rbu_wgrad_args* a);
int rbu_wgrad_halo_launch(const rbu_wgrad_args* a, void* workspace, cudaStream_t stream);
// wgrad_gemm.cu: the split-K reduction of the weight-gradient partials
void rbu_wgrad_reduce_launch(const float* partial, int ksplit, int Mtot, int taps, int Ntot, float* out, int accumulate,
                             cudaStream_t stream);

extern "C" size_t rbu_conv_stats_floats(int Ncols);
