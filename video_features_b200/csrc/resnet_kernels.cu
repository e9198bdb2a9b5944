// Memory-bound kernels of the ResNet path (resnet.cu): the fused transform + stem pack, the stem max pool, the
// residual add + ReLU and the global average pool.  Activations are single-fp16 channels-last rows of zero-bordered
// volumes (Vol2, conv2d.h); the precision policy is in DESIGN.md §4.6.
#include "common.cuh"
#include "internal.h"
#include "resnet_kernels.h"

namespace vf {

namespace {

inline unsigned nb(int64_t total, int threads) { return unsigned((total + threads - 1) / threads); }

// Phase volume of the 7x7 stride-2 pad-3 stem: out[b][hq][wq][(ph*2+pw)*4 + c] = x[2(hq-2)+ph][2(wq-2)+pw][c] in fp16,
// 16 channels per row (12 used), zero outside the 224x224 frame (the conv's own padding).
// u8 source: resized frames [n][Hr][Wr][3]; the 224 crop at (cy, cx), channel order reversed when swap_rb, and
// ToTensor + Normalize in fp32 (imagenet_norm) -- every source byte is read once.
// fp32 source: frames already normalised, [n][3][224][224].
template <bool U8>
__global__ void stem_pack_kernel(const void* __restrict__ src, int n, int Hr, int Wr, int cy, int cx, int swap_rb,
                                 __half* __restrict__ out) {
    constexpr int Q = RESNET_STEM_Q;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(n) * Q * Q;
    if (idx >= total) return;
    const int wq = int(idx % Q), hq = int((idx / Q) % Q), b = int(idx / (int64_t(Q) * Q));
    __align__(16) __half vals[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) vals[i] = __float2half_rn(0.f);
#pragma unroll
    for (int ph = 0; ph < 2; ++ph)
#pragma unroll
        for (int pw = 0; pw < 2; ++pw) {
            const int y = 2 * (hq - 2) + ph, x = 2 * (wq - 2) + pw;
            if (y < 0 || y >= 224 || x < 0 || x >= 224) continue;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float v;
                if (U8) {
                    const uint8_t* p = static_cast<const uint8_t*>(src) + ((int64_t(b) * Hr + cy + y) * Wr + cx + x) * 3;
                    v = imagenet_norm(__ldg(p + (swap_rb ? 2 - c : c)), c);
                } else {
                    v = __ldg(static_cast<const float*>(src) + ((int64_t(b) * 3 + c) * 224 + y) * 224 + x);
                }
                vals[(ph * 2 + pw) * 4 + c] = __float2half_rn(v);
            }
        }
    uint4* o = reinterpret_cast<uint4*>(out + idx * 16);
    o[0] = reinterpret_cast<const uint4*>(vals)[0];
    o[1] = reinterpret_cast<const uint4*>(vals)[1];
}

// 3x3 stride-2 pad-1 max pool from the stem output (valid region of vi) into the valid region of the border-1
// volume vo; vo's border rows are written as zeros.  Padding is skipped rather than read as -inf: the input is
// post-ReLU (>= 0) and every window holds at least one valid element, so the result equals torch's -inf padding
// (and equally a zero padding).
__global__ void maxpool_kernel(const __half* __restrict__ in, Vol2 vi, int C, __half* __restrict__ out, Vol2 vo) {
    const int cg = C >> 3;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(vo.n) * vo.Hp * vo.Wp * cg;
    if (idx >= total) return;
    const int c8 = int(idx % cg);
    const int64_t pos = idx / cg;
    const int wq = int(pos % vo.Wp), hq = int((pos / vo.Wp) % vo.Hp), b = int(pos / (int64_t(vo.Wp) * vo.Hp));
    uint4 r = make_uint4(0, 0, 0, 0);
    if (hq >= vo.h0 && hq < vo.h1 && wq >= vo.w0 && wq < vo.w1) {
        __half2 m[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) m[j] = __float2half2_rn(0.f);
        const int y0 = 2 * (hq - vo.h0) - 1, x0 = 2 * (wq - vo.w0) - 1;
        for (int dy = 0; dy < 3; ++dy) {
            const int y = y0 + dy;
            if (y < 0 || y >= vi.h1 - vi.h0) continue;
            for (int dx = 0; dx < 3; ++dx) {
                const int x = x0 + dx;
                if (x < 0 || x >= vi.w1 - vi.w0) continue;
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(
                    in + ((int64_t(b) * vi.Hp + y + vi.h0) * vi.Wp + x + vi.w0) * C + c8 * 8));
                const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
                for (int j = 0; j < 4; ++j) m[j] = __hmax2(m[j], h[j]);
            }
        }
        r = *reinterpret_cast<const uint4*>(m);
    }
    *reinterpret_cast<uint4*>(out + pos * C + c8 * 8) = r;
}

// out = relu(a + b) in fp32, rounded once to fp16, on valid positions; border rows zero.  out may alias a or b.
__global__ void add_relu_kernel(const __half* a, const __half* bsrc, __half* out, Vol2 v, int C) {
    const int cg = C >> 3;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * v.Hp * v.Wp * cg;
    if (idx >= total) return;
    const int c8 = int(idx % cg);
    const int64_t pos = idx / cg;
    const int wq = int(pos % v.Wp), hq = int((pos / v.Wp) % v.Hp);
    const int64_t off = pos * C + c8 * 8;
    if (hq < v.h0 || hq >= v.h1 || wq < v.w0 || wq >= v.w1) {
        *reinterpret_cast<uint4*>(out + off) = make_uint4(0, 0, 0, 0);
        return;
    }
    const uint4 av = *reinterpret_cast<const uint4*>(a + off), bv = *reinterpret_cast<const uint4*>(bsrc + off);
    const __half *pa = reinterpret_cast<const __half*>(&av), *pb = reinterpret_cast<const __half*>(&bv);
    __align__(16) __half o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = __float2half_rn(fmaxf(__half2float(pa[j]) + __half2float(pb[j]), 0.f));
    *reinterpret_cast<uint4*>(out + off) = *reinterpret_cast<const uint4*>(o);
}

// out[b][c] = mean over the valid region of channel c; one thread per (b, c), rows summed in a fixed order in fp32.
__global__ void avgpool_kernel(const __half* __restrict__ in, Vol2 v, int C, float* __restrict__ out) {
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= int64_t(v.n) * C) return;
    const int c = int(idx % C), b = int(idx / C);
    float s = 0.f;
    for (int y = v.h0; y < v.h1; ++y)
        for (int x = v.w0; x < v.w1; ++x) s += __half2float(in[((int64_t(b) * v.Hp + y) * v.Wp + x) * C + c]);
    out[idx] = s / float((v.h1 - v.h0) * (v.w1 - v.w0));
}

}  // namespace

#define LAUNCH_CHECK() do { VF_CUDA(cudaGetLastError()); return VF_OK; } while (0)

int resnet_stem_pack_u8(const uint8_t* src, int n, int Hr, int Wr, int cy, int cx, int swap_rb, __half* out,
                        cudaStream_t s) {
    const int64_t total = int64_t(n) * RESNET_STEM_Q * RESNET_STEM_Q;
    stem_pack_kernel<true><<<nb(total, 256), 256, 0, s>>>(src, n, Hr, Wr, cy, cx, swap_rb, out);
    LAUNCH_CHECK();
}
int resnet_stem_pack_f32(const float* src, int n, __half* out, cudaStream_t s) {
    const int64_t total = int64_t(n) * RESNET_STEM_Q * RESNET_STEM_Q;
    stem_pack_kernel<false><<<nb(total, 256), 256, 0, s>>>(src, n, 224, 224, 0, 0, 0, out);
    LAUNCH_CHECK();
}
int resnet_maxpool(const __half* in, const Vol2& vi, int C, __half* out, const Vol2& vo, cudaStream_t s) {
    maxpool_kernel<<<nb(vo.rows() * (C / 8), 256), 256, 0, s>>>(in, vi, C, out, vo);
    LAUNCH_CHECK();
}
int resnet_add_relu(const __half* a, const __half* b, __half* out, const Vol2& v, int C, cudaStream_t s) {
    add_relu_kernel<<<nb(v.rows() * (C / 8), 256), 256, 0, s>>>(a, b, out, v, C);
    LAUNCH_CHECK();
}
int resnet_avgpool(const __half* in, const Vol2& v, int C, float* out, cudaStream_t s) {
    avgpool_kernel<<<nb(int64_t(v.n) * C, 256), 256, 0, s>>>(in, v, C, out);
    LAUNCH_CHECK();
}

}  // namespace vf
