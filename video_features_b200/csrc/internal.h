// Host-side internals shared by the translation units of libvfeat.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/vfeat.h"

namespace vf {

// thread-local last-error text behind vf_last_error()
void set_error(const char* fmt, ...);
int fail(int code, const char* fmt, ...);

#define VF_CUDA(expr)                                                                       \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess)                                                              \
            return vf::fail(VF_ERR_CUDA, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,      \
                            cudaGetErrorString(_e));                                        \
    } while (0)
#define VF_TRY(expr)                  \
    do {                              \
        int _s = (expr);              \
        if (_s != VF_OK) return _s;   \
    } while (0)

// ---- tensor maps (driver entry point fetched at run time; the library does not link libcuda).
// 2-D row-major tensor of 2- or 4-byte elements, 128-byte-swizzled boxes of box_rows x (128 / elem_bytes) columns.
int make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t rows, uint64_t cols,
                 uint64_t row_pitch_bytes, uint32_t box_rows, uint32_t box_cols);

// ---- GEMM: D[M,N] = act(A[M,K] . B[N,K]^T * scale[n] + bias[n]), fp16 operands, fp32 accumulate (tcgen05)
struct GemmEpi {
    void* out;              // fp16 or fp32, row pitch ldo elements, 16-byte aligned rows
    const float* bias;      // [N] or null
    const float* scale;     // [N] or null
    int ldo;
    int out_f32;            // 0: fp16 out, 1: fp32 out
    int act;                // VF_ACT_*
    int split_off;          // fp16 out only: > 0 writes the result as a split-fp16 pair, hi at column n and
                            // lo = fp16(v - hi) at column split_off + n of the same row (0: plain fp16)
    int accumulate;         // fp32 out only: 1 = out += result (a TMA reduction in the L2; every element is added exactly
                            // once, so the sum is deterministic) -- the residual-stream update of the ViT blocks
};
int gemm_f16(const __half* A, int lda, const __half* B, int ldb, int M, int N, int K, const GemmEpi& ep,
             cudaStream_t stream);

// ---- shifted-row ("implicit GEMM") convolution on the same kernel.
// Activations live channels-last in a zero-bordered volume [n][Tp][Hp][Wp][C] flattened to P rows of C channels.
// A filter tap (dt,dh,dw) is then a constant row shift of the whole matrix, and because consecutive w positions are
// consecutive rows, the kw taps of one (dt,dh) form ONE contiguous run of kw*C elements: the A operand of tap j is
// the overlapping-row view  A_j[p, 0:k_per_tap] = X[(p + tap_off[j]) * C : ... + k_per_tap].
// Rows whose position lies outside the valid region [t0,t1)x[h0,h1)x[w0,w1) are written as zeros (they are the
// zero padding the next layer reads).
struct ConvGeom {
    int ntaps;          // number of (dt,dh) taps (1 for a 1x1x1 conv)
    int k_per_tap;      // contiguous K elements per tap (kw * C)
    int tap_off[64];    // row shift of each tap (includes the shift to the first kw tap)
    int nsplit;         // 1, or 2: weights are a hi+lo fp16 pair, Wt = [hi (ntaps*k_per_tap) | lo (same)] along K; every
                        // A tile is loaded once and multiplied with both (A.W_hi + A.W_lo)
    unsigned long long lo_mask;   // nsplit == 2 only: bit kk set = K block kk of every tap holds only lo halves of split-fp16
                        // activations (or unused columns): the W_lo pass is skipped there (a_lo.w_lo is below fp32 eps)
    int row0;           // leading guard rows: row m of the matrix is position m - row0 of the volume (rows < row0 are zeroed)
    int mask;           // 1: zero the rows outside the valid region
    int Tp, Hp, Wp;     // padded volume extents (rows per sample = Tp*Hp*Wp)
    int t0, t1, h0, h1, w0, w1;
};
// X: [P, C] fp16 (row pitch C), Wt: [N, ntaps*k_per_tap] fp16, output rows = P
int conv_gemm_f16(const __half* X, int C, int64_t P, const __half* Wt, int N, const ConvGeom& g, const GemmEpi& ep,
                  cudaStream_t stream);
// ---- QKV projection fused with the 50-token attention (csrc/attn_gemm.cu): h [n_frames*50, 768] fp16 -> att [.., heads*64]
// w_perm: in_proj rows regrouped per head, row h*192 + part*64 + d = in_proj row part*768 + h*64 + d (bias likewise)
int qkv_attention(const __half* h, int lda, const __half* w_perm, const float* bias_perm, __half* att, int n_frames, int heads,
                  cudaStream_t stream);
int device_sm_count();
int gemm_profile(int enable);
bool gemm_profile_on();   // event-bracketed launches cannot be captured into a graph: callers fall back to eager
int gemm_profile_read(double* ms, int64_t* launches, double* flops);

// ---- elementwise / reduction kernels
// patch = 32 (ViT-B/32: [n*49, 3072] patch rows) or 16 (ViT-B/16: [n*196, 768])
int launch_clip_patchify(const uint8_t* src, int n, int src_h, int src_w, int crop_y, int crop_x, __half* patches,
                         int patch, cudaStream_t s);
int launch_clip_patchify_f32(const float* src_chw, int n, __half* patches, int patch, cudaStream_t s);
int launch_clip_normalize_f32(const uint8_t* src, int n, int src_h, int src_w, int crop_y, int crop_x, float* dst_chw,
                              cudaStream_t s);
// the same with torchvision's ImageNet mean / std (ResNet); swap_rb reads BGR frames as RGB
int launch_imagenet_normalize_f32(const uint8_t* src, int n, int src_h, int src_w, int crop_y, int crop_x, int swap_rb,
                                  float* dst_chw, cudaStream_t s);
// x (+= y) ; out = LayerNorm(x) -- rows of 768 fp32.  y may be null; write_x stores the summed residual stream back.
int launch_add_layernorm(float* x, int64_t x_row_stride, const __half* y, int64_t y_row_stride, int write_x,
                         const float* gamma, const float* beta, void* out, int64_t out_row_stride, int out_f32, int rows,
                         cudaStream_t s);
// ViT embedding rows: token 0 = cls_pos0, token t>0 = emb[frame*(tokens-1) + t-1] + pos[t]; x = ln_pre(row) (fp32)
int launch_embed_layernorm(const float* emb, const float* pos, const float* cls_pos0, const float* gamma,
                           const float* beta, float* x, int n_frames, int tokens, cudaStream_t s);
// self-attention per (frame, head) on a [n_frames*tokens, 3*heads*64] QKV matrix: tokens == 50 or 65..208
int launch_attention(const __half* qkv, __half* out, int n_frames, int tokens, int heads, cudaStream_t s);
int launch_resample(const uint8_t* src, int n, int in_h, int in_w, uint8_t* tmp, uint8_t* dst, int out_h, int out_w,
                    const int* kh_bounds, const int* kh_coef, int kh_size, const int* kv_bounds, const int* kv_coef,
                    int kv_size, cudaStream_t s);

// host: Pillow-compatible resize (coefficient tables built in float64, cached on the device per geometry)
int resize_u8(const uint8_t* src, int n, int in_h, int in_w, uint8_t* dst, int out_h, int out_w, int filter,
              uint8_t* tmp, cudaStream_t s);
// torchvision CenterCrop offset: int(round((dim - crop) / 2.0)), Python round-half-to-even
int center_crop_offset(int dim, int crop);

}  // namespace vf
