// Memory-bound kernels of the CLIP path: frame transform (normalise / patchify), LayerNorm,
// 50-token attention, and the Pillow-compatible fixed-point resample.  All are HBM/L2-bound
// byte-and-float shuffles: 128-bit accesses, warp-shuffle reductions, no tensor cores.
#include <atomic>

#include "common.cuh"
#include "internal.h"

namespace vf {

namespace {

// clip.clip._transform Normalize constants (third-party openai/CLIP), float32-rounded like torch does
__constant__ float kClipMean[3] = {0.48145466f, 0.4578275f, 0.40821073f};
__constant__ float kClipStd[3] = {0.26862954f, 0.26130258f, 0.27577711f};

__device__ __forceinline__ float clip_norm(uint8_t v, int c) {
    // ToTensor: float32(v) / 255 ; Normalize: (x - mean) / std -- IEEE fp32 ops, same order as torchvision
    return __fdiv_rn(__fsub_rn(__fdiv_rn(float(v), 255.0f), kClipMean[c]), kClipStd[c]);
}

// uint8 HWC frames (cropped window 224x224 at (cy,cx)) -> fp16 patch matrix [n*G*G, 3*PS*PS] (G = 224/PS patches a side:
// [n*49, 3072] for ViT-B/32, [n*196, 768] for ViT-B/16), column = c*PS*PS + ky*PS + kx (the natural flattening of
// conv1.weight[768,3,PS,PS]).  One thread: 16 pixels (48 B in, 3 x 32 B out).
template <int PS>
__global__ void clip_patchify_u8_kernel(const uint8_t* __restrict__ src, int n, int src_h, int src_w, int cy, int cx,
                                        __half* __restrict__ out) {
    constexpr int G = 224 / PS, PP = PS * PS;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(n) * 224 * 14;
    if (idx >= total) return;
    const int xg = int(idx % 14);
    const int y = int((idx / 14) % 224);
    const int b = int(idx / (14 * 224));
    const uint8_t* p = src + ((int64_t(b) * src_h + cy + y) * src_w + cx + xg * 16) * 3;
    __align__(16) uint8_t px[48];
    if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
        const uint4* p4 = reinterpret_cast<const uint4*>(p);
        uint4* d4 = reinterpret_cast<uint4*>(px);
        d4[0] = __ldg(p4);
        d4[1] = __ldg(p4 + 1);
        d4[2] = __ldg(p4 + 2);
    } else {
#pragma unroll
        for (int i = 0; i < 48; ++i) px[i] = __ldg(p + i);
    }
    const int py = y / PS, ky = y % PS, pxi = (xg * 16) / PS, kx0 = (xg * 16) % PS;
    __half* orow = out + (int64_t(b) * (G * G) + py * G + pxi) * (3 * PP) + ky * PS + kx0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        uint32_t pk[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
            pk[i] = pack_half2(clip_norm(px[(2 * i) * 3 + c], c), clip_norm(px[(2 * i + 1) * 3 + c], c));
        uint4* o4 = reinterpret_cast<uint4*>(orow + c * PP);
        o4[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        o4[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
    }
}

// fp32 CHW frames (already transformed, what encode_image receives) -> fp16 patch matrix. 8 px / thread.
template <int PS>
__global__ void clip_patchify_f32_kernel(const float* __restrict__ src, int n, __half* __restrict__ out) {
    constexpr int G = 224 / PS, PP = PS * PS;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(n) * 3 * 224 * 28;
    if (idx >= total) return;
    const int xg = int(idx % 28);
    const int y = int((idx / 28) % 224);
    const int c = int((idx / (28 * 224)) % 3);
    const int b = int(idx / (28 * 224 * 3));
    const float4* p = reinterpret_cast<const float4*>(src + ((int64_t(b) * 3 + c) * 224 + y) * 224 + xg * 8);
    const float4 a = __ldg(p), d = __ldg(p + 1);
    const int py = y / PS, ky = y % PS, pxi = (xg * 8) / PS, kx0 = (xg * 8) % PS;
    __half* o = out + (int64_t(b) * (G * G) + py * G + pxi) * (3 * PP) + c * PP + ky * PS + kx0;
    *reinterpret_cast<uint4*>(o) =
        make_uint4(pack_half2(a.x, a.y), pack_half2(a.z, a.w), pack_half2(d.x, d.y), pack_half2(d.z, d.w));
}

struct ClipNorm {
    __device__ static float apply(uint8_t v, int c) { return clip_norm(v, c); }
};
struct ImageNetNorm {
    __device__ static float apply(uint8_t v, int c) { return imagenet_norm(v, c); }
};

// uint8 HWC (crop window) -> fp32 CHW normalised: the tensor the reference feeds the network. 4 px / thread.
// swap_rb: read the source's channels in reverse order (BGR frames -> RGB values)
template <class Norm>
__global__ void normalize_f32_kernel(const uint8_t* __restrict__ src, int n, int src_h, int src_w, int cy, int cx,
                                     int swap_rb, float* __restrict__ dst) {
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(n) * 224 * 56;
    if (idx >= total) return;
    const int xg = int(idx % 56);
    const int y = int((idx / 56) % 224);
    const int b = int(idx / (56 * 224));
    const uint8_t* p = src + ((int64_t(b) * src_h + cy + y) * src_w + cx + xg * 4) * 3;
    uint8_t px[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) px[i] = __ldg(p + i);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int sc = swap_rb ? 2 - c : c;
        float4 v = make_float4(Norm::apply(px[sc], c), Norm::apply(px[3 + sc], c), Norm::apply(px[6 + sc], c),
                               Norm::apply(px[9 + sc], c));
        *reinterpret_cast<float4*>(dst + ((int64_t(b) * 3 + c) * 224 + y) * 224 + xg * 4) = v;
    }
}

// LayerNorm over rows of 768 fp32 (eps 1e-5, biased variance): one warp per row, the row lives in registers
// (6 float4 per lane), mean and variance by warp shuffles (two-pass, no E[x^2]-E[x]^2 cancellation).
struct Row768 {
    float4 v[6];
};
__device__ __forceinline__ void ln768_write(const Row768& r, int lane, const float* __restrict__ gamma,
                                            const float* __restrict__ beta, void* out_row, int out_f32) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 6; ++i) s += (r.v[i].x + r.v[i].y) + (r.v[i].z + r.v[i].w);
    const float mean = warp_sum(s) * (1.0f / 768.0f);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const float a = r.v[i].x - mean, b = r.v[i].y - mean, c = r.v[i].z - mean, d = r.v[i].w - mean;
        q += (a * a + b * b) + (c * c + d * d);
    }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / 768.0f) + 1e-5f);
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const int col = (lane + 32 * i) * 4;
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + col));
        const float4 bb = __ldg(reinterpret_cast<const float4*>(beta + col));
        float4 y;
        y.x = (r.v[i].x - mean) * rstd * g.x + bb.x;
        y.y = (r.v[i].y - mean) * rstd * g.y + bb.y;
        y.z = (r.v[i].z - mean) * rstd * g.z + bb.z;
        y.w = (r.v[i].w - mean) * rstd * g.w + bb.w;
        if (out_f32) *reinterpret_cast<float4*>(reinterpret_cast<float*>(out_row) + col) = y;
        else *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(out_row) + col) =
                 make_uint2(pack_half2(y.x, y.y), pack_half2(y.z, y.w));
    }
}

// LayerNorm of the residual stream, optionally fused with its update:  HAS_Y: x += y first (y = the previous GEMM's
// output as an fp16 increment; x itself stays fp32), out = LN(x).  Without y (the GEMM epilogue already added its result
// into x with a TMA reduction) a pass reads 4 and writes 2 bytes per element.  Compile-time variants: the plain one keeps
// no y registers live and fits 6 blocks of 8 warps per SM without spilling.
#ifndef VF_LN_BLOCKS
#define VF_LN_BLOCKS 5      // resident blocks per SM the register allocation targets (6 spills 40 bytes per thread)
#endif
template <bool HAS_Y, bool OUT_F32>
__global__ void __launch_bounds__(256, VF_LN_BLOCKS) add_layernorm768_kernel(float* __restrict__ x, int64_t row_stride,
                                        const __half* __restrict__ y, int64_t y_row_stride, int write_x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                        void* out, int64_t out_row_stride, int rows) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + warp;
    if (row >= rows) return;
    float* xr = x + int64_t(row) * row_stride;
    Row768 r;
#pragma unroll
    for (int i = 0; i < 6; ++i) r.v[i] = *reinterpret_cast<const float4*>(xr + (lane + 32 * i) * 4);
    if (HAS_Y) {
        const __half* yr = y + int64_t(row) * y_row_stride;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const uint2 raw = __ldg(reinterpret_cast<const uint2*>(yr + (lane + 32 * i) * 4));
            const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
            const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
            r.v[i].x += a.x; r.v[i].y += a.y; r.v[i].z += b.x; r.v[i].w += b.y;
        }
        if (write_x) {
#pragma unroll
            for (int i = 0; i < 6; ++i) *reinterpret_cast<float4*>(xr + (lane + 32 * i) * 4) = r.v[i];
        }
    }
    void* orow = OUT_F32 ? static_cast<void*>(reinterpret_cast<float*>(out) + int64_t(row) * out_row_stride)
                         : static_cast<void*>(reinterpret_cast<__half*>(out) + int64_t(row) * out_row_stride);
    ln768_write(r, lane, gamma, beta, orow, OUT_F32 ? 1 : 0);
}

// ViT token assembly fused with ln_pre: row (frame, t): t == 0 -> class_embedding + pos[0] (precomputed),
// t > 0 -> patch embedding row (frame*(tokens-1) + t-1) + pos[t];  x = ln_pre(row) in fp32.
__global__ void __launch_bounds__(256, 6) embed_layernorm768_kernel(const float* __restrict__ emb, const float* __restrict__ pos,
                                          const float* __restrict__ cls_pos0, const float* __restrict__ gamma,
                                          const float* __restrict__ beta, float* __restrict__ x, int rows, int tokens) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + warp;
    if (row >= rows) return;
    const int frame = row / tokens, t = row - frame * tokens;
    Row768 r;
    if (t == 0) {
#pragma unroll
        for (int i = 0; i < 6; ++i) r.v[i] = __ldg(reinterpret_cast<const float4*>(cls_pos0 + (lane + 32 * i) * 4));
    } else {
        const float* er = emb + (int64_t(frame) * (tokens - 1) + (t - 1)) * 768;
        const float* pr = pos + t * 768;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(er + (lane + 32 * i) * 4));
            const float4 p = __ldg(reinterpret_cast<const float4*>(pr + (lane + 32 * i) * 4));
            r.v[i] = make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w);
        }
    }
    ln768_write(r, lane, gamma, beta, x + int64_t(row) * 768, 1);
}

// Self-attention for one (frame, head): S = 50 tokens, head_dim 64, no mask.  q is scaled by 1/8 after the
// in-projection (torch nn.MultiheadAttention semantics; applied here to the fp32 scores, which is the same
// arithmetic since 1/8 is a power of two).  The two contractions are 64x64x64 after padding -- far too small for a
// tcgen05 tile, so they run on warp-level mma.sync (m16n8k16, fp16 in / fp32 accumulate): one block of 4 warps
// per (frame, head), warp w owns query rows 16w..16w+15.  Q, K, V are staged once in shared memory with 16-byte
// cp.async (row pitch 144 B: conflict-free ldmatrix), fragments come from ldmatrix (.trans for V), the softmax
// lives in the accumulator fragments (fp32) with quad shuffles, and O goes back through shared memory so that the
// global stores are full 128-byte rows.
constexpr int ATT_S = 50, ATT_D = 64, ATT_LD = 72;

__device__ __forceinline__ void mma16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t* r, const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t* r, const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}

__global__ void __launch_bounds__(128) attention50_kernel(const __half* __restrict__ qkv, __half* __restrict__ out,
                                                          int heads) {
    __shared__ __align__(16) __half Qs[64][ATT_LD];   // [query][dim]; reused for O
    __shared__ __align__(16) __half Ks[64][ATT_LD];   // [key][dim]
    __shared__ __align__(16) __half Vs[64][ATT_LD];   // [key][dim]
    const int frame = blockIdx.x / heads, head = blockIdx.x % heads;
    const int width = heads * ATT_D;
    const int ld = 3 * width;
    const int64_t row0 = int64_t(frame) * ATT_S;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;

    // stage Q, K, V rows 0..49 (3 x 400 16-byte chunks); zero K/V rows 50..63 (0 * garbage must stay 0 in P.V)
    for (int i = tid; i < 3 * ATT_S * 8; i += 128) {
        const int m = i / (ATT_S * 8), rem = i - m * (ATT_S * 8);
        const int r = rem >> 3, seg = rem & 7;
        const __half* src = qkv + (row0 + r) * ld + m * width + head * ATT_D + seg * 8;
        __half* dst = (m == 0 ? &Qs[r][seg * 8] : m == 1 ? &Ks[r][seg * 8] : &Vs[r][seg * 8]);
        cp_async16(dst, src);
    }
    for (int i = tid; i < 2 * 14 * 8; i += 128) {
        const int m = i / (14 * 8), rem = i - m * (14 * 8);
        const int r = ATT_S + (rem >> 3), seg = rem & 7;
        *reinterpret_cast<uint4*>(m == 0 ? &Ks[r][seg * 8] : &Vs[r][seg * 8]) = make_uint4(0, 0, 0, 0);
    }
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    const int q0 = warp * 16;
    // S = Q K^T : A fragments of this warp's 16 query rows (4 dim steps), B fragments of K per key tile
    uint32_t aq[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) ldsm_x4(aq[ks], &Qs[q0 + (lane & 15)][ks * 16 + (lane >> 4) * 8]);
    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
        for (int kp = 0; kp < 2; ++kp) {   // two dim steps per ldmatrix.x4
            uint32_t bk[4];
            ldsm_x4(bk, &Ks[nt * 8 + (lane & 7)][kp * 32 + (lane >> 3) * 8]);
            mma16816(s[nt], aq[2 * kp], bk[0], bk[1]);
            mma16816(s[nt], aq[2 * kp + 1], bk[2], bk[3]);
        }
    }
    // softmax over the 50 valid keys; this thread holds rows q0+g (regs 0,1) and q0+g+8 (regs 2,3)
    const float sc = 0.125f * 1.4426950408889634f;   // 1/sqrt(64) * log2(e)
    float m_lo = -INFINITY, m_hi = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const bool valid = nt * 8 + 2 * t + j < ATT_S;
            s[nt][j] = valid ? s[nt][j] * sc : -INFINITY;
            s[nt][2 + j] = valid ? s[nt][2 + j] * sc : -INFINITY;
            m_lo = fmaxf(m_lo, s[nt][j]);
            m_hi = fmaxf(m_hi, s[nt][2 + j]);
        }
    }
    m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 1));
    m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 2));
    m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 1));
    m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 2));
    float sum_lo = 0.f, sum_hi = 0.f;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            s[nt][j] = exp2f(s[nt][j] - m_lo);          // exp2f(-inf) == 0 for the padded keys
            s[nt][2 + j] = exp2f(s[nt][2 + j] - m_hi);
            sum_lo += s[nt][j];
            sum_hi += s[nt][2 + j];
        }
    }
    sum_lo += __shfl_xor_sync(0xffffffffu, sum_lo, 1);
    sum_lo += __shfl_xor_sync(0xffffffffu, sum_lo, 2);
    sum_hi += __shfl_xor_sync(0xffffffffu, sum_hi, 1);
    sum_hi += __shfl_xor_sync(0xffffffffu, sum_hi, 2);
    const float inv_lo = 1.0f / sum_lo, inv_hi = 1.0f / sum_hi;

    // O = P V : accumulator fragments of S become the A fragments of P (normalised in fp32 first)
    uint32_t pa[4][4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        pa[kk][0] = pack_half2(s[2 * kk][0] * inv_lo, s[2 * kk][1] * inv_lo);
        pa[kk][1] = pack_half2(s[2 * kk][2] * inv_hi, s[2 * kk][3] * inv_hi);
        pa[kk][2] = pack_half2(s[2 * kk + 1][0] * inv_lo, s[2 * kk + 1][1] * inv_lo);
        pa[kk][3] = pack_half2(s[2 * kk + 1][2] * inv_hi, s[2 * kk + 1][3] * inv_hi);
    }
    __syncwarp();   // every lane's ldmatrix reads of this warp's Q rows are done before they are overwritten with O
#pragma unroll
    for (int np = 0; np < 4; ++np) {        // two dim tiles per ldmatrix.x4.trans
        float o0[4] = {0.f, 0.f, 0.f, 0.f}, o1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            uint32_t bv[4];
            ldsm_x4_trans(bv, &Vs[kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8][np * 16 + (lane >> 4) * 8]);
            mma16816(o0, pa[kk], bv[0], bv[1]);
            mma16816(o1, pa[kk], bv[2], bv[3]);
        }
        *reinterpret_cast<uint32_t*>(&Qs[q0 + g][np * 16 + 2 * t]) = pack_half2(o0[0], o0[1]);
        *reinterpret_cast<uint32_t*>(&Qs[q0 + g + 8][np * 16 + 2 * t]) = pack_half2(o0[2], o0[3]);
        *reinterpret_cast<uint32_t*>(&Qs[q0 + g][np * 16 + 8 + 2 * t]) = pack_half2(o1[0], o1[1]);
        *reinterpret_cast<uint32_t*>(&Qs[q0 + g + 8][np * 16 + 8 + 2 * t]) = pack_half2(o1[2], o1[3]);
    }
    __syncwarp();
    // this warp's 16 output rows, 128 B each, as 16-byte stores (8 lanes cover one row)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = q0 + i * 4 + (lane >> 3), seg = lane & 7;
        if (r < ATT_S)
            *reinterpret_cast<uint4*>(out + (row0 + r) * width + head * ATT_D + seg * 8) =
                *reinterpret_cast<const uint4*>(&Qs[r][seg * 8]);
    }
}

// The same attention for longer sequences (ViT-B/16: S = 197 tokens): NT 16-key tiles cover the padded sequence, one
// block of NW warps per (frame, head), a warp owns query tiles w, w+NW, ...  K, V and Q of the head live in dynamic
// shared memory (3 x 16*NT rows x 144 B).  The keys are taken in two halves with a running (max, sum) -- the usual
// online softmax -- so that a thread holds the scores of half a row (52 registers at NT = 13), two blocks fit an SM and
// one block's staging overlaps the other's arithmetic.  P is rounded to fp16 before normalisation (values in [0,1]),
// the 1/sum factor is applied to the fp32 output.
template <int KT0, int KTN>
__device__ __forceinline__ void attention_keys(const __half (*Ks)[ATT_LD], const __half (*Vs)[ATT_LD], const uint32_t (*aq)[4],
                                               float (*o)[4], float& m_lo, float& m_hi, float& l_lo, float& l_hi, int S,
                                               int lane) {
    const int t = lane & 3;
    const float sc = 0.125f * 1.4426950408889634f;   // 1/sqrt(64) * log2(e)
    float s[2 * KTN][4];
#pragma unroll
    for (int nt = 0; nt < 2 * KTN; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
        for (int kp = 0; kp < 2; ++kp) {
            uint32_t bk[4];
            ldsm_x4(bk, &Ks[KT0 * 16 + nt * 8 + (lane & 7)][kp * 32 + (lane >> 3) * 8]);
            mma16816(s[nt], aq[2 * kp], bk[0], bk[1]);
            mma16816(s[nt], aq[2 * kp + 1], bk[2], bk[3]);
        }
    }
    float n_lo = m_lo, n_hi = m_hi;
#pragma unroll
    for (int nt = 0; nt < 2 * KTN; ++nt) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const bool valid = KT0 * 16 + nt * 8 + 2 * t + j < S;
            s[nt][j] = valid ? s[nt][j] * sc : -INFINITY;
            s[nt][2 + j] = valid ? s[nt][2 + j] * sc : -INFINITY;
            n_lo = fmaxf(n_lo, s[nt][j]);
            n_hi = fmaxf(n_hi, s[nt][2 + j]);
        }
    }
    n_lo = fmaxf(n_lo, __shfl_xor_sync(0xffffffffu, n_lo, 1));
    n_lo = fmaxf(n_lo, __shfl_xor_sync(0xffffffffu, n_lo, 2));
    n_hi = fmaxf(n_hi, __shfl_xor_sync(0xffffffffu, n_hi, 1));
    n_hi = fmaxf(n_hi, __shfl_xor_sync(0xffffffffu, n_hi, 2));
    // rescale what has been accumulated under the old maximum (exp2f(-inf) == 0 on the first half)
    const float r_lo = exp2f(m_lo - n_lo), r_hi = exp2f(m_hi - n_hi);
    m_lo = n_lo; m_hi = n_hi;
    l_lo *= r_lo; l_hi *= r_hi;
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[i][0] *= r_lo; o[i][1] *= r_lo; o[i][2] *= r_hi; o[i][3] *= r_hi; }
#pragma unroll
    for (int nt = 0; nt < 2 * KTN; ++nt) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            s[nt][j] = exp2f(s[nt][j] - m_lo);
            s[nt][2 + j] = exp2f(s[nt][2 + j] - m_hi);
            l_lo += s[nt][j];
            l_hi += s[nt][2 + j];
        }
    }
#pragma unroll
    for (int kk = 0; kk < KTN; ++kk) {           // 16 keys per step: P fragments straight from the score fragments
        uint32_t pa[4];
        pa[0] = pack_half2(s[2 * kk][0], s[2 * kk][1]);
        pa[1] = pack_half2(s[2 * kk][2], s[2 * kk][3]);
        pa[2] = pack_half2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        pa[3] = pack_half2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
        for (int np = 0; np < 4; ++np) {
            uint32_t bv[4];
            ldsm_x4_trans(bv, &Vs[(KT0 + kk) * 16 + (lane & 7) + ((lane >> 3) & 1) * 8][np * 16 + (lane >> 4) * 8]);
            mma16816(o[2 * np], pa, bv[0], bv[1]);
            mma16816(o[2 * np + 1], pa, bv[2], bv[3]);
        }
    }
}

template <int NT, int NW>
__global__ void __launch_bounds__(NW * 32, 2) attention_long_kernel(const __half* __restrict__ qkv, __half* __restrict__ out,
                                                                     int heads, int S) {
    constexpr int SP = NT * 16, H0 = (NT + 1) / 2, H1 = NT - H0;
    extern __shared__ __align__(16) uint8_t att_smem[];
    __half (*Qs)[ATT_LD] = reinterpret_cast<__half (*)[ATT_LD]>(att_smem);
    __half (*Ks)[ATT_LD] = Qs + SP;
    __half (*Vs)[ATT_LD] = Ks + SP;
    const int frame = blockIdx.x / heads, head = blockIdx.x % heads;
    const int width = heads * ATT_D;
    const int ld = 3 * width;
    const int64_t row0 = int64_t(frame) * S;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;

    for (int i = tid; i < 3 * S * 8; i += NW * 32) {
        const int m = i / (S * 8), rem = i - m * (S * 8);
        const int r = rem >> 3, seg = rem & 7;
        const __half* src = qkv + (row0 + r) * ld + m * width + head * ATT_D + seg * 8;
        cp_async16(m == 0 ? &Qs[r][seg * 8] : m == 1 ? &Ks[r][seg * 8] : &Vs[r][seg * 8], src);
    }
    const int pad = SP - S;                   // zero rows S..SP-1 of Q (finite scores), K and V (0 * garbage stays 0)
    for (int i = tid; i < 3 * pad * 8; i += NW * 32) {
        const int m = i / (pad * 8), rem = i - m * (pad * 8);
        const int r = S + (rem >> 3), seg = rem & 7;
        *reinterpret_cast<uint4*>(m == 0 ? &Qs[r][seg * 8] : m == 1 ? &Ks[r][seg * 8] : &Vs[r][seg * 8]) = make_uint4(0, 0, 0, 0);
    }
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    for (int mt = warp; mt * 16 < S; mt += NW) {
        const int q0 = mt * 16;
        uint32_t aq[4][4];
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) ldsm_x4(aq[ks], &Qs[q0 + (lane & 15)][ks * 16 + (lane >> 4) * 8]);
        float o[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
        float m_lo = -INFINITY, m_hi = -INFINITY, l_lo = 0.f, l_hi = 0.f;
        attention_keys<0, H0>(Ks, Vs, aq, o, m_lo, m_hi, l_lo, l_hi, S, lane);
        attention_keys<H0, H1>(Ks, Vs, aq, o, m_lo, m_hi, l_lo, l_hi, S, lane);
        l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 1);
        l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 2);
        l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 1);
        l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 2);
        const float inv_lo = 1.0f / l_lo, inv_hi = 1.0f / l_hi;
        __syncwarp();   // this warp's ldmatrix reads of its own Q rows are done; they become the O staging rows
#pragma unroll
        for (int np = 0; np < 4; ++np) {
            *reinterpret_cast<uint32_t*>(&Qs[q0 + g][np * 16 + 2 * t]) = pack_half2(o[2 * np][0] * inv_lo, o[2 * np][1] * inv_lo);
            *reinterpret_cast<uint32_t*>(&Qs[q0 + g + 8][np * 16 + 2 * t]) = pack_half2(o[2 * np][2] * inv_hi, o[2 * np][3] * inv_hi);
            *reinterpret_cast<uint32_t*>(&Qs[q0 + g][np * 16 + 8 + 2 * t]) = pack_half2(o[2 * np + 1][0] * inv_lo, o[2 * np + 1][1] * inv_lo);
            *reinterpret_cast<uint32_t*>(&Qs[q0 + g + 8][np * 16 + 8 + 2 * t]) = pack_half2(o[2 * np + 1][2] * inv_hi, o[2 * np + 1][3] * inv_hi);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = q0 + i * 4 + (lane >> 3), seg = lane & 7;
            if (r < S)
                *reinterpret_cast<uint4*>(out + (row0 + r) * width + head * ATT_D + seg * 8) =
                    *reinterpret_cast<const uint4*>(&Qs[r][seg * 8]);
        }
    }
}

// Pillow ImagingResampleHorizontal_8bpc / Vertical_8bpc (third-party Pillow, libImaging/Resample.c), 3 channels:
//   acc = 2^21 + sum_i px[i] * k[i]  (int32) ;  out = clip8(acc >> 22)
// Frames are byte streams whose rows (w*3 bytes) are rarely 16-byte multiples, so both passes move CONTIGUOUS SPANS of
// rows through shared memory: the span is fetched / written back with 128-bit accesses on its 16-byte-aligned body (the
// few head / tail bytes go one by one), staged at the same offset modulo 16 as in global memory, and the per-pixel
// arithmetic reads and writes bytes in shared memory only.
__device__ __forceinline__ uint8_t clip8(int acc) {
    const int v = acc >> 22;
    return uint8_t(v < 0 ? 0 : (v > 255 ? 255 : v));
}
// smem[off .. off+n) <- g[0 .. n)  with off == (address of g) mod 16
__device__ __forceinline__ void span_load(uint8_t* smem, const uint8_t* __restrict__ g, int64_t n, int tid, int nthreads) {
    const int off = int(reinterpret_cast<uintptr_t>(g) & 15);
    const int head = off ? min(int64_t(16 - off), n) : 0;
    const int64_t body = (n - head) >> 4;
    for (int i = tid; i < head; i += nthreads) smem[off + i] = __ldg(g + i);
    const uint4* g4 = reinterpret_cast<const uint4*>(g + head);
    uint4* s4 = reinterpret_cast<uint4*>(smem + off + head);
    for (int64_t i = tid; i < body; i += nthreads) s4[i] = __ldg(g4 + i);
    const int64_t done = head + (body << 4);
    for (int64_t i = done + tid; i < n; i += nthreads) smem[off + i] = __ldg(g + i);
}
__device__ __forceinline__ void span_store(uint8_t* __restrict__ g, const uint8_t* smem, int64_t n, int tid, int nthreads) {
    const int off = int(reinterpret_cast<uintptr_t>(g) & 15);
    const int head = off ? min(int64_t(16 - off), n) : 0;
    const int64_t body = (n - head) >> 4;
    for (int i = tid; i < head; i += nthreads) g[i] = smem[off + i];
    uint4* g4 = reinterpret_cast<uint4*>(g + head);
    const uint4* s4 = reinterpret_cast<const uint4*>(smem + off + head);
    for (int64_t i = tid; i < body; i += nthreads) g4[i] = s4[i];
    const int64_t done = head + (body << 4);
    for (int64_t i = done + tid; i < n; i += nthreads) g[i] = smem[off + i];
}

// horizontal pass: a block owns `rows_per_block` consecutive rows of the flattened (n * in_h) row list
__global__ void __launch_bounds__(256) resample_h_kernel(const uint8_t* __restrict__ src, int64_t total_rows, int in_w,
                                                         uint8_t* __restrict__ dst, int out_w, const int* __restrict__ bounds,
                                                         const int* __restrict__ coef, int ksize, int rows_per_block,
                                                         int in_cap) {
    extern __shared__ __align__(16) uint8_t rs_smem[];
    const int64_t row0 = int64_t(blockIdx.x) * rows_per_block;
    const int rows = int(min(int64_t(rows_per_block), total_rows - row0));
    const uint8_t* gin = src + row0 * in_w * 3;
    uint8_t* gout = dst + row0 * out_w * 3;
    uint8_t* sin = rs_smem;
    uint8_t* sout = rs_smem + in_cap;                       // in_cap: multiple of 16 >= rows_per_block*in_w*3 + 16
    span_load(sin, gin, int64_t(rows) * in_w * 3, threadIdx.x, blockDim.x);
    __syncthreads();
    const uint8_t* pin = sin + (reinterpret_cast<uintptr_t>(gin) & 15);
    uint8_t* pout = sout + (reinterpret_cast<uintptr_t>(gout) & 15);
    for (int idx = threadIdx.x; idx < rows * out_w; idx += blockDim.x) {
        const int r = idx / out_w, xx = idx - r * out_w;
        const int xmin = __ldg(bounds + 2 * xx), cnt = __ldg(bounds + 2 * xx + 1);
        const int* k = coef + int64_t(xx) * ksize;
        const uint8_t* p = pin + (r * in_w + xmin) * 3;
        int s0 = 1 << 21, s1 = 1 << 21, s2 = 1 << 21;
        for (int i = 0; i < cnt; ++i) {
            const int kv = __ldg(k + i);
            s0 += int(p[3 * i]) * kv;
            s1 += int(p[3 * i + 1]) * kv;
            s2 += int(p[3 * i + 2]) * kv;
        }
        uint8_t* o = pout + idx * 3;
        o[0] = clip8(s0);
        o[1] = clip8(s1);
        o[2] = clip8(s2);
    }
    __syncthreads();
    span_store(gout, sout, int64_t(rows) * out_w * 3, threadIdx.x, blockDim.x);
}

// vertical pass: a block owns `rows_per_block` output rows of ONE frame and the input rows they read ([lo, hi), at
// most in_rows_cap of them); every byte column of a row is an independent 1-D filter, so channels need no special case
__global__ void __launch_bounds__(256) resample_v_kernel(const uint8_t* __restrict__ src, int in_h, int w3,
                                                         uint8_t* __restrict__ dst, int out_h, const int* __restrict__ bounds,
                                                         const int* __restrict__ coef, int ksize, int rows_per_block,
                                                         int blocks_per_frame, int in_cap) {
    extern __shared__ __align__(16) uint8_t rs_smem[];
    const int b = blockIdx.x / blocks_per_frame;
    const int yy0 = (blockIdx.x - b * blocks_per_frame) * rows_per_block;
    const int rows = min(rows_per_block, out_h - yy0);
    const int lo = __ldg(bounds + 2 * yy0);
    const int hi = __ldg(bounds + 2 * (yy0 + rows - 1)) + __ldg(bounds + 2 * (yy0 + rows - 1) + 1);
    const uint8_t* gin = src + (int64_t(b) * in_h + lo) * w3;
    uint8_t* gout = dst + (int64_t(b) * out_h + yy0) * w3;
    uint8_t* sin = rs_smem;
    uint8_t* sout = rs_smem + in_cap;
    span_load(sin, gin, int64_t(hi - lo) * w3, threadIdx.x, blockDim.x);
    __syncthreads();
    const uint8_t* pin = sin + (reinterpret_cast<uintptr_t>(gin) & 15);
    uint8_t* pout = sout + (reinterpret_cast<uintptr_t>(gout) & 15);
    for (int idx = threadIdx.x; idx < rows * w3; idx += blockDim.x) {
        const int r = idx / w3, j = idx - r * w3;
        const int yy = yy0 + r;
        const int ymin = __ldg(bounds + 2 * yy), cnt = __ldg(bounds + 2 * yy + 1);
        const int* k = coef + int64_t(yy) * ksize;
        const uint8_t* p = pin + (ymin - lo) * w3 + j;
        int acc = 1 << 21;
        for (int i = 0; i < cnt; ++i) acc += int(p[i * w3]) * __ldg(k + i);
        pout[idx] = clip8(acc);
    }
    __syncthreads();
    span_store(gout, sout, int64_t(rows) * w3, threadIdx.x, blockDim.x);
}

inline unsigned blocks_for(int64_t total, int threads) { return unsigned((total + threads - 1) / threads); }

}  // namespace

int launch_clip_patchify(const uint8_t* src, int n, int src_h, int src_w, int crop_y, int crop_x, __half* patches,
                         int patch, cudaStream_t s) {
    const int64_t total = int64_t(n) * 224 * 14;
    if (patch == 32)
        clip_patchify_u8_kernel<32><<<blocks_for(total, 256), 256, 0, s>>>(src, n, src_h, src_w, crop_y, crop_x, patches);
    else if (patch == 16)
        clip_patchify_u8_kernel<16><<<blocks_for(total, 256), 256, 0, s>>>(src, n, src_h, src_w, crop_y, crop_x, patches);
    else
        return fail(VF_ERR_UNSUPPORTED, "patchify: patch size %d (32 and 16 are built)", patch);
    VF_CUDA(cudaGetLastError());
    return VF_OK;
}
int launch_clip_patchify_f32(const float* src_chw, int n, __half* patches, int patch, cudaStream_t s) {
    const int64_t total = int64_t(n) * 3 * 224 * 28;
    if (patch == 32)
        clip_patchify_f32_kernel<32><<<blocks_for(total, 256), 256, 0, s>>>(src_chw, n, patches);
    else if (patch == 16)
        clip_patchify_f32_kernel<16><<<blocks_for(total, 256), 256, 0, s>>>(src_chw, n, patches);
    else
        return fail(VF_ERR_UNSUPPORTED, "patchify: patch size %d (32 and 16 are built)", patch);
    VF_CUDA(cudaGetLastError());
    return VF_OK;
}
int launch_clip_normalize_f32(const uint8_t* src, int n, int src_h, int src_w, int crop_y, int crop_x, float* dst_chw,
                              cudaStream_t s) {
    const int64_t total = int64_t(n) * 224 * 56;
    normalize_f32_kernel<ClipNorm><<<blocks_for(total, 256), 256, 0, s>>>(src, n, src_h, src_w, crop_y, crop_x, 0, dst_chw);
    VF_CUDA(cudaGetLastError());
    return VF_OK;
}
int launch_imagenet_normalize_f32(const uint8_t* src, int n, int src_h, int src_w, int crop_y, int crop_x, int swap_rb,
                                  float* dst_chw, cudaStream_t s) {
    const int64_t total = int64_t(n) * 224 * 56;
    normalize_f32_kernel<ImageNetNorm><<<blocks_for(total, 256), 256, 0, s>>>(src, n, src_h, src_w, crop_y, crop_x, swap_rb,
                                                                             dst_chw);
    VF_CUDA(cudaGetLastError());
    return VF_OK;
}
int launch_add_layernorm(float* x, int64_t x_row_stride, const __half* y, int64_t y_row_stride, int write_x,
                         const float* gamma, const float* beta, void* out, int64_t out_row_stride, int out_f32, int rows,
                         cudaStream_t s) {
    const int warps = 8;
    const dim3 grid((rows + warps - 1) / warps), block(warps * 32);
#define VF_LN(HY, F32) add_layernorm768_kernel<HY, F32><<<grid, block, 0, s>>>(x, x_row_stride, y, y_row_stride, write_x, gamma, \
                                                                             beta, out, out_row_stride, rows)
    if (y != nullptr) { if (out_f32) VF_LN(true, true); else VF_LN(true, false); }
    else              { if (out_f32) VF_LN(false, true); else VF_LN(false, false); }
#undef VF_LN
    VF_CUDA(cudaGetLastError());
    return VF_OK;
}
int launch_embed_layernorm(const float* emb, const float* pos, const float* cls_pos0, const float* gamma,
                           const float* beta, float* x, int n_frames, int tokens, cudaStream_t s) {
    const int warps = 8, rows = n_frames * tokens;
    embed_layernorm768_kernel<<<(rows + warps - 1) / warps, warps * 32, 0, s>>>(emb, pos, cls_pos0, gamma, beta, x, rows, tokens);
    VF_CUDA(cudaGetLastError());
    return VF_OK;
}
int launch_attention(const __half* qkv, __half* out, int n_frames, int tokens, int heads, cudaStream_t s) {
    if (tokens == ATT_S) {
        attention50_kernel<<<n_frames * heads, 128, 0, s>>>(qkv, out, heads);
    } else if (tokens > 64 && tokens <= 208) {
        constexpr int NT = 13, NW = 8;                       // 208 padded keys; 13 query tiles over 8 warps
        constexpr int kSmem = 3 * NT * 16 * ATT_LD * int(sizeof(__half));
        static std::atomic<bool> attr_done[64];
        int dev = 0;
        VF_CUDA(cudaGetDevice(&dev));
        if (dev >= 0 && dev < 64 && !attr_done[dev].load(std::memory_order_acquire)) {
            VF_CUDA(cudaFuncSetAttribute(attention_long_kernel<NT, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
            attr_done[dev].store(true, std::memory_order_release);
        }
        attention_long_kernel<NT, NW><<<n_frames * heads, NW * 32, kSmem, s>>>(qkv, out, heads, tokens);
    } else {
        return fail(VF_ERR_UNSUPPORTED, "attention: %d tokens (50 and 65..208 are built)", tokens);
    }
    VF_CUDA(cudaGetLastError());
    return VF_OK;
}
int launch_resample(const uint8_t* src, int n, int in_h, int in_w, uint8_t* tmp, uint8_t* dst, int out_h, int out_w,
                    const int* kh_bounds, const int* kh_coef, int kh_size, const int* kv_bounds, const int* kv_coef,
                    int kv_size, cudaStream_t s) {
    // Pillow order: horizontal pass first (rounded to uint8), then vertical; a pass is skipped when the
    // axis size is unchanged (ImagingResample: need_horizontal / need_vertical).
    const bool need_h = out_w != in_w, need_v = out_h != in_h;
    const uint8_t* cur = src;
    constexpr int kMaxSmem = 200 * 1024;
    static std::atomic<bool> attr_done[64];
    int dev = 0;
    VF_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_done[dev].load(std::memory_order_acquire)) {
        VF_CUDA(cudaFuncSetAttribute(resample_h_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
        VF_CUDA(cudaFuncSetAttribute(resample_v_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
        attr_done[dev].store(true, std::memory_order_release);
    }
    auto round16 = [](int64_t v) { return int((v + 15) / 16 * 16); };
    if (need_h) {
        uint8_t* hdst = need_v ? tmp : dst;
        const int64_t total_rows = int64_t(n) * in_h;
        // rows per block: as many as fit ~48 KB of staging (in + out), at least 1, at most 16
        int rpb = int(48 * 1024 / (int64_t(in_w + out_w) * 3));
        rpb = rpb < 1 ? 1 : (rpb > 16 ? 16 : rpb);
        const int in_cap = round16(int64_t(rpb) * in_w * 3 + 16), out_cap = round16(int64_t(rpb) * out_w * 3 + 16);
        if (in_cap + out_cap > kMaxSmem) return fail(VF_ERR_UNSUPPORTED, "resize: rows of %d px do not fit shared memory", in_w);
        const unsigned blocks = unsigned((total_rows + rpb - 1) / rpb);
        resample_h_kernel<<<blocks, 256, in_cap + out_cap, s>>>(cur, total_rows, in_w, hdst, out_w, kh_bounds, kh_coef, kh_size,
                                                               rpb, in_cap);
        VF_CUDA(cudaGetLastError());
        cur = hdst;
    }
    if (need_v) {
        const int w3 = out_w * 3;
        // output rows per block: 8 unless the rows are very wide; the input span of a block is bounded by
        // rows * scale + filter taps (+1 for the fractional start)
        const double scale = double(in_h) / double(out_h);
        int rpb = 8;
        int in_rows_cap = 0, in_cap = 0, out_cap = 0;
        for (;; rpb = rpb / 2) {
            in_rows_cap = int(rpb * (scale > 1.0 ? scale : 1.0)) + kv_size + 2;
            if (in_rows_cap > in_h) in_rows_cap = in_h;
            in_cap = round16(int64_t(in_rows_cap) * w3 + 16);
            out_cap = round16(int64_t(rpb) * w3 + 16);
            if (in_cap + out_cap <= 96 * 1024 || rpb == 1) break;
        }
        if (in_cap + out_cap > kMaxSmem) return fail(VF_ERR_UNSUPPORTED, "resize: rows of %d px do not fit shared memory", out_w);
        const int bpf = (out_h + rpb - 1) / rpb;
        resample_v_kernel<<<unsigned(n) * bpf, 256, in_cap + out_cap, s>>>(cur, in_h, w3, dst, out_h, kv_bounds, kv_coef, kv_size,
                                                                          rpb, bpf, in_cap);
        VF_CUDA(cudaGetLastError());
    } else if (!need_h) {
        VF_CUDA(cudaMemcpyAsync(dst, src, size_t(n) * in_h * in_w * 3, cudaMemcpyDeviceToDevice, s));
    }
    return VF_OK;
}

}  // namespace vf
