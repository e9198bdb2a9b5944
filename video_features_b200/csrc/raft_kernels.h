// Launchers of the RAFT memory-bound kernels (raft_kernels.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "conv2d.h"   // Vol2

namespace vf {

// Row layout of the GRU operand buffers hx / qx (768 columns = 12 K blocks of 64, each purely hi or purely lo):
//   [h_hi 0..127 | h_lo 128..255 | inp_hi 256..383 | inp_lo 384..511 | motion_hi 512..637, flow_hi 638..639 |
//    motion_lo 640..765, flow_lo 766..767]
// (the GRU input is cat[h, inp, motion-encoder output (126), flow (2)]: the flow takes the two spare slots of the
// 128-wide motion block; the motion conv stores only its first 126 columns.)
constexpr int RAFT_HX = 768, RAFT_HX_MOTION = 512, RAFT_HX_FLOW = 638, RAFT_HX_LO = 128;
// correlation features (324 = 4 levels x 81): [hi 324 + 60 zero | lo 324 + 60 zero]
constexpr int RAFT_CF = 768, RAFT_CF_LO = 384;

int raft_input_pack(const void* img, int is_u8, int chw, int n, int Hs, int Ws, int pad_top, int pad_left, int H, int W,
                    __half* out, int Hq, int Wq, cudaStream_t s);
int raft_instnorm_stats(const float* x, const Vol2& v, int C, double* stats, cudaStream_t s);
int raft_instnorm_apply(const float* a, const double* a_stats, const __half* res_h, const float* res_raw,
                        const double* res_stats, __half* out, const Vol2& v, int C, cudaStream_t s);
int raft_add_relu(const __half* a, const __half* b, __half* out, const Vol2& v, int C, cudaStream_t s);
int raft_gather_valid(const __half* in, const Vol2& v, int C, int ld, __half* out, cudaStream_t s);
int raft_corr_pool(float* corr, int64_t rows, int ld, int off_in, int Hi, int Wi, int off_out, cudaStream_t s);
int raft_corr_lookup(const float* corr, int ld, const float* coords, int n, int H8, int W8, __half* out, const Vol2& vo,
                     int out_ld, cudaStream_t s);
int raft_corr_operands(const float* f, const Vol2& v, int P8, __half* A, __half* B, cudaStream_t s);
int raft_cnet_split(const float* cnet, const Vol2& vi, __half* hx, __half* qx, float* h32, const Vol2& vo, int ld,
                    cudaStream_t s);
int raft_gru_rh(const __half* hx, const float* h32, const float* zr, __half* qx, const Vol2& v, int ld, cudaStream_t s);
int raft_gru_update(__half* hx, float* h32, const float* zr, const float* q, const Vol2& v, int ld, cudaStream_t s);
int raft_coords_update(float* coords1, const float* delta, __half* hx, __half* qx, __half* flow8, const Vol2& v, int ld,
                       cudaStream_t s);
int raft_flow_fill(const __half* flow8, __half* hx, const Vol2& v, int ld, cudaStream_t s);
int raft_upsample_flow(const float* coords1, const float* mask, const Vol2& v, int n, int H8, int W8, int oy, int ox,
                       int Ho, int Wo, float* flow_up, cudaStream_t s);
int raft_unpack2d_f32(const float* in, const Vol2& v, int ld, int c0, int cc, float* out, cudaStream_t s);
int raft_unpack2d(const __half* in, const Vol2& v, int ld, int c0, int cc, int lo_off, float* out, cudaStream_t s);

}  // namespace vf
