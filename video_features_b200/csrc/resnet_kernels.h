// Launchers of the ResNet memory-bound kernels (resnet_kernels.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "conv2d.h"   // Vol2

namespace vf {

// side of the stem's phase volume: 112 output positions + 2 border rows before + 1 after (the 7x7/2 taps reach
// positions q-2 .. q+1 of the phase grid)
constexpr int RESNET_STEM_Q = 115;

int resnet_stem_pack_u8(const uint8_t* src, int n, int Hr, int Wr, int cy, int cx, int swap_rb, __half* out,
                        cudaStream_t s);
int resnet_stem_pack_f32(const float* src, int n, __half* out, cudaStream_t s);
int resnet_maxpool(const __half* in, const Vol2& vi, int C, __half* out, const Vol2& vo, cudaStream_t s);
int resnet_add_relu(const __half* a, const __half* b, __half* out, const Vol2& v, int C, cudaStream_t s);
int resnet_avgpool(const __half* in, const Vol2& v, int C, float* out, cudaStream_t s);

}  // namespace vf
