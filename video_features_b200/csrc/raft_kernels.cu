// Memory-bound kernels of the RAFT path.  Activations are channels-last fp16 rows of zero-bordered 2-D volumes
// [n][Hp][Wp][C] (see raft.cu for the geometry); coordinates / flow / correlation volume are fp32.
#include "common.cuh"
#include "internal.h"
#include "raft_kernels.h"

namespace vf {

namespace {

// split-fp16 representation of an fp32 value: v ~= hi + lo with |lo| <= 2^-11 |hi|
__device__ __forceinline__ void split_half(float v, __half& hi, __half& lo) {
    hi = __float2half_rn(v);
    lo = __float2half_rn(v - __half2float(hi));
}

inline unsigned nb(int64_t total, int threads) { return unsigned((total + threads - 1) / threads); }

// images [n][H][W][3] (uint8 or fp32 in [0,255]) -> 2*(x/255) - 1 (raft.py:118-119) -> phase volume for the 7x7
// stride-2 pad-3 stem: out[hq][wq][((ph*2+pw)*4 + c)] = x[2(hq-2)+ph][2(wq-2)+pw][c] as a split-fp16 pair:
// 32 channels = [16 hi (12 used) | 16 lo].
// (Hs, Ws) is the source frame; (H, W) the /8-padded frame with the source at (pad_top, pad_left): InputPadder's
// replicate padding (raft.py:36-37) is a coordinate clamp.
template <typename TIn>
__global__ void raft_input_pack_kernel(const TIn* __restrict__ img, int n, int Hs, int Ws, int pad_top, int pad_left,
                                       int H, int W, int chw_layout, __half* __restrict__ out, int Hq, int Wq) {
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(n) * Hq * Wq;
    if (idx >= total) return;
    const int wq = int(idx % Wq), hq = int((idx / Wq) % Hq), b = int(idx / (int64_t(Wq) * Hq));
    __align__(16) __half vals[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) vals[i] = __float2half_rn(0.f);
#pragma unroll
    for (int ph = 0; ph < 2; ++ph)
#pragma unroll
        for (int pw = 0; pw < 2; ++pw) {
            const int yp = 2 * (hq - 2) + ph, xp = 2 * (wq - 2) + pw;
            if (yp < 0 || yp >= H || xp < 0 || xp >= W) continue;       // the conv's own zero padding
            const int y = min(max(yp - pad_top, 0), Hs - 1), x = min(max(xp - pad_left, 0), Ws - 1);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float v = chw_layout ? float(img[((int64_t(b) * 3 + c) * Hs + y) * Ws + x])
                                           : float(img[((int64_t(b) * Hs + y) * Ws + x) * 3 + c]);
                split_half(__fsub_rn(__fmul_rn(2.0f, __fdiv_rn(v, 255.0f)), 1.0f), vals[(ph * 2 + pw) * 4 + c],
                           vals[16 + (ph * 2 + pw) * 4 + c]);
            }
        }
    uint4* o = reinterpret_cast<uint4*>(out + idx * 32);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = reinterpret_cast<const uint4*>(vals)[i];
}

// InstanceNorm2d statistics: per (sample, channel) sum and sum of squares over the valid region.  grid (H, n): one block
// per image row, block = C * S threads (S position phases per channel); fp32 partials per thread over <= W/S values, the
// S partials and the rows are combined in double.
__global__ void instnorm_stats_kernel(const float* __restrict__ x, Vol2 v, int C, double* __restrict__ stats) {
    __shared__ double red[2][256];
    const int b = blockIdx.y, y = blockIdx.x;
    const int c = threadIdx.x % C, sub = threadIdx.x / C, S = blockDim.x / C;
    const int W = v.w1 - v.w0;
    const float* row = x + ((int64_t(b) * v.Hp + y + v.h0) * v.Wp + v.w0) * C + c;
    float fs = 0.f, fss = 0.f;
    for (int xw = sub; xw < W; xw += S) {
        const float t = row[int64_t(xw) * C];
        fs += t;
        fss = fmaf(t, t, fss);
    }
    red[0][threadIdx.x] = double(fs);
    red[1][threadIdx.x] = double(fss);
    __syncthreads();
    if (sub == 0) {
        double s = 0.0, ss = 0.0;
        for (int j = 0; j < S; ++j) { s += red[0][j * C + c]; ss += red[1][j * C + c]; }
        atomicAdd(&stats[(int64_t(b) * C + c) * 2], s);
        atomicAdd(&stats[(int64_t(b) * C + c) * 2 + 1], ss);
    }
}

// The raw conv outputs that feed InstanceNorm are kept in fp32 (an fp16 copy would lose |mean|/|std| bits in the
// mean subtraction), and the normalised activations -- the A operands of the next conv -- are written as split-fp16
// pairs: row = [hi C | lo C] (the conv weights are duplicated over both halves).
// y = relu(IN(a))                                                    (res_h == res_raw == nullptr)
// y = relu(res_h + relu(IN(a)))                                      stride-1 ResidualBlock tail (res_h: split x)
// y = relu(IN(res_raw) + relu(IN(a)))                                stride-2 ResidualBlock tail (norm3(downsample))
// Every position of the volume is written; border positions get zeros (the next conv's padding).  8 channels/thread.
__global__ void instnorm_apply_kernel(const float* __restrict__ a, const double* __restrict__ a_stats,
                                      const __half* __restrict__ res_h, const float* __restrict__ res_raw,
                                      const double* __restrict__ res_stats, __half* __restrict__ out, Vol2 v, int C) {
    const int cg = C >> 3;
    const int H = v.h1 - v.h0, W = v.w1 - v.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * v.Hp * v.Wp * cg;
    if (idx >= total) return;
    const int c8 = int(idx % cg);
    const int64_t pos = idx / cg;
    const int wq = int(pos % v.Wp), hq = int((pos / v.Wp) % v.Hp), b = int(pos / (int64_t(v.Wp) * v.Hp));
    const int64_t off = pos * C + c8 * 8;              // fp32 raw rows: pitch C
    const int64_t off2 = pos * (2 * C) + c8 * 8;       // split rows: pitch 2C
    if (hq < v.h0 || hq >= v.h1 || wq < v.w0 || wq >= v.w1) {
        *reinterpret_cast<uint4*>(out + off2) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(out + off2 + C) = make_uint4(0, 0, 0, 0);
        return;
    }
    const double inv_cnt = 1.0 / (double(H) * double(W));     // one divide per thread; the 8 channels multiply
    float av[8], rv[8];
    *reinterpret_cast<float4*>(av) = *reinterpret_cast<const float4*>(a + off);
    *reinterpret_cast<float4*>(av + 4) = *reinterpret_cast<const float4*>(a + off + 4);
    if (res_raw) {
        *reinterpret_cast<float4*>(rv) = *reinterpret_cast<const float4*>(res_raw + off);
        *reinterpret_cast<float4*>(rv + 4) = *reinterpret_cast<const float4*>(res_raw + off + 4);
    } else if (res_h) {
        const uint4 rh = *reinterpret_cast<const uint4*>(res_h + off2);
        const uint4 rl = *reinterpret_cast<const uint4*>(res_h + off2 + C);
        const __half* hh = reinterpret_cast<const __half*>(&rh);
        const __half* hl = reinterpret_cast<const __half*>(&rl);
#pragma unroll
        for (int j = 0; j < 8; ++j) rv[j] = __half2float(hh[j]) + __half2float(hl[j]);
    }
    __align__(16) __half oh[8], ol[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int c = c8 * 8 + j;
        const double m = a_stats[(int64_t(b) * C + c) * 2] * inv_cnt;
        const double var = a_stats[(int64_t(b) * C + c) * 2 + 1] * inv_cnt - m * m;
        float y0 = float((double(av[j]) - m)) * rsqrtf(float(var) + 1e-5f);
        y0 = fmaxf(y0, 0.f);
        if (res_raw) {
            const double rm = res_stats[(int64_t(b) * C + c) * 2] * inv_cnt;
            const double rvv = res_stats[(int64_t(b) * C + c) * 2 + 1] * inv_cnt - rm * rm;
            y0 = fmaxf(float(double(rv[j]) - rm) * rsqrtf(float(rvv) + 1e-5f) + y0, 0.f);
        } else if (res_h) {
            y0 = fmaxf(rv[j] + y0, 0.f);
        }
        split_half(y0, oh[j], ol[j]);
    }
    *reinterpret_cast<uint4*>(out + off2) = *reinterpret_cast<const uint4*>(oh);
    *reinterpret_cast<uint4*>(out + off2 + C) = *reinterpret_cast<const uint4*>(ol);
}

// out = relu(a + b) on valid positions, all three stored as split-fp16 rows [hi C | lo C] (batch-norm encoder: the
// norms are folded into the conv epilogues, which write the split pairs themselves)
__global__ void add_relu_kernel(const __half* __restrict__ a, const __half* __restrict__ bsrc, __half* __restrict__ out,
                                Vol2 v, int C) {
    const int cg = C >> 3;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * v.Hp * v.Wp * cg;
    if (idx >= total) return;
    const int c8 = int(idx % cg);
    const int64_t pos = idx / cg;
    const int wq = int(pos % v.Wp), hq = int((pos / v.Wp) % v.Hp);
    const int64_t off = pos * (2 * C) + c8 * 8;
    if (hq < v.h0 || hq >= v.h1 || wq < v.w0 || wq >= v.w1) {
        *reinterpret_cast<uint4*>(out + off) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(out + off + C) = make_uint4(0, 0, 0, 0);
        return;
    }
    const uint4 ah = *reinterpret_cast<const uint4*>(a + off), al = *reinterpret_cast<const uint4*>(a + off + C);
    const uint4 bh = *reinterpret_cast<const uint4*>(bsrc + off), bl = *reinterpret_cast<const uint4*>(bsrc + off + C);
    const __half *pah = reinterpret_cast<const __half*>(&ah), *pal = reinterpret_cast<const __half*>(&al);
    const __half *pbh = reinterpret_cast<const __half*>(&bh), *pbl = reinterpret_cast<const __half*>(&bl);
    __align__(16) __half oh[8], ol[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float x = (__half2float(pah[j]) + __half2float(pal[j])) + (__half2float(pbh[j]) + __half2float(pbl[j]));
        split_half(fmaxf(x, 0.f), oh[j], ol[j]);
    }
    *reinterpret_cast<uint4*>(out + off) = *reinterpret_cast<const uint4*>(oh);
    *reinterpret_cast<uint4*>(out + off + C) = *reinterpret_cast<const uint4*>(ol);
}

// valid rows of a bordered volume -> dense [n][H*W][C]
__global__ void gather_valid_kernel(const __half* __restrict__ in, Vol2 v, int C, int ld, __half* __restrict__ out) {
    const int cg = C >> 3;
    const int H = v.h1 - v.h0, W = v.w1 - v.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * H * W * cg;
    if (idx >= total) return;
    const int c8 = int(idx % cg);
    const int64_t pos = idx / cg;
    const int xw = int(pos % W), y = int((pos / W) % H), b = int(pos / (int64_t(W) * H));
    const int64_t off = ((int64_t(b) * v.Hp + y + v.h0) * v.Wp + xw + v.w0) * ld + c8 * 8;
    *reinterpret_cast<uint4*>(out + pos * C + c8 * 8) = *reinterpret_cast<const uint4*>(in + off);
}

// fnet features (fp32 rows of a border-1 volume, 256 ch) -> the two operand forms of the 3-term split correlation
//   corr = f1 . f2 ~= f1_hi.f2_hi + f1_lo.f2_hi + f1_hi.f2_lo :  A rows = [hi | lo | hi], B rows = [hi | hi | lo]  (K = 768)
// so the all-pairs volume is exact to ~2^-22 instead of carrying two fp16 operand roundings.  Dense [n][P8][768].
__global__ void corr_operands_kernel(const float* __restrict__ f, Vol2 v, int P8, __half* __restrict__ A,
                                     __half* __restrict__ B) {
    const int H = v.h1 - v.h0, W = v.w1 - v.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * H * W * 32;       // 8 channels per thread
    if (idx >= total) return;
    const int c8 = int(idx % 32);
    const int64_t pos = idx / 32;
    const int xw = int(pos % W), y = int((pos / W) % H), b = int(pos / (int64_t(W) * H));
    const float* src = f + ((int64_t(b) * v.Hp + y + v.h0) * v.Wp + xw + v.w0) * 256 + c8 * 8;
    float fv[8];
    *reinterpret_cast<float4*>(fv) = *reinterpret_cast<const float4*>(src);
    *reinterpret_cast<float4*>(fv + 4) = *reinterpret_cast<const float4*>(src + 4);
    __align__(16) __half hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) split_half(fv[j], hi[j], lo[j]);
    const int64_t row = (int64_t(b) * P8 + y * W + xw) * 768 + c8 * 8;
    const uint4 H4 = *reinterpret_cast<const uint4*>(hi), L4 = *reinterpret_cast<const uint4*>(lo);
    *reinterpret_cast<uint4*>(A + row) = H4;
    *reinterpret_cast<uint4*>(A + row + 256) = L4;
    *reinterpret_cast<uint4*>(A + row + 512) = H4;
    *reinterpret_cast<uint4*>(B + row) = H4;
    *reinterpret_cast<uint4*>(B + row + 256) = H4;
    *reinterpret_cast<uint4*>(B + row + 512) = L4;
}

// correlation pyramid: level l+1 = avg_pool2d(level l, 2, 2) over the (h2, w2) axes of every query row
// (corr.py:24-27; floor sizes).  corr row layout: [lvl0 H*W | lvl1 | lvl2 | lvl3] floats, pitch `ld`.
__global__ void corr_pool_kernel(float* __restrict__ corr, int64_t rows, int ld, int off_in, int Hi, int Wi, int off_out) {
    const int Ho = Hi / 2, Wo = Wi / 2;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = rows * Ho * Wo;
    if (idx >= total) return;
    const int xo = int(idx % Wo), yo = int((idx / Wo) % Ho);
    const int64_t r = idx / (int64_t(Wo) * Ho);
    const float* p = corr + r * ld + off_in + (2 * yo) * Wi + 2 * xo;
    corr[r * ld + off_out + yo * Wo + xo] = 0.25f * ((p[0] + p[1]) + (p[Wi] + p[Wi + 1]));
}

// CorrBlock.__call__ (corr.py:29-50): for every query position and pyramid level, the 9x9 window of bilinear
// samples (zero outside the map, align_corners=True pixel coordinates) around coords/2^l.  The window is the
// reference's TRANSPOSED one: output channel l*81 + i*9 + j samples (x + i-4, y + j-4).
// One warp per (query, level): the 10x10 integer neighbourhood is fetched once, the 81 blends come from it.
__global__ void corr_lookup_kernel(const float* __restrict__ corr, int ld, const float* __restrict__ coords, int n,
                                   int H8, int W8, __half* __restrict__ out, Vol2 vo, int out_ld) {
    const int lane = threadIdx.x & 31;
    const int64_t wid = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int64_t total = int64_t(n) * H8 * W8 * 4;
    if (wid >= total) return;
    const int lvl = int(wid & 3);
    const int64_t q = wid >> 2;                      // b*H8*W8 + y*W8 + x
    const int x0 = int(q % W8), y0 = int((q / W8) % H8), b = int(q / (int64_t(W8) * H8));
    // level offsets inside a corr row: level 0 occupies P8 = roundup(H8*W8, 8) columns (the GEMM's N), the pooled levels
    // follow densely (raft.cu: lvl_off)
    int Hl = H8, Wl = W8, off = 0;
    for (int l = 0; l < lvl; ++l) { off += (l == 0) ? ((Hl * Wl + 7) & ~7) : Hl * Wl; Hl >>= 1; Wl >>= 1; }
    const float inv = 1.0f / float(1 << lvl);
    const float cx = coords[q * 2] * inv, cy = coords[q * 2 + 1] * inv;
    const float fx0 = floorf(cx), fy0 = floorf(cy);
    const float ax = cx - fx0, ay = cy - fy0;
    const int ix = int(fx0) - 4, iy = int(fy0) - 4;     // top-left of the 10x10 neighbourhood
    const float* row = corr + q * ld + off;
    __shared__ float nbuf[8][104];
    float* nbr = nbuf[(threadIdx.x >> 5)];
    for (int i = lane; i < 100; i += 32) {
        const int yy = iy + i / 10, xx = ix + i % 10;
        nbr[i] = (yy >= 0 && yy < Hl && xx >= 0 && xx < Wl) ? row[yy * Wl + xx] : 0.f;
    }
    __syncwarp();
    const int64_t orow = (int64_t(b) * vo.Hp + y0 + vo.h0) * vo.Wp + x0 + vo.w0;
    __half* o = out + orow * out_ld + lvl * 81;
    for (int k = lane; k < 81; k += 32) {
        const int i = k / 9, j = k % 9;                 // i offsets x, j offsets y (transposed window)
        const float v00 = nbr[j * 10 + i], v01 = nbr[j * 10 + i + 1];
        const float v10 = nbr[(j + 1) * 10 + i], v11 = nbr[(j + 1) * 10 + i + 1];
        const float v = (1.f - ay) * ((1.f - ax) * v00 + ax * v01) + ay * ((1.f - ax) * v10 + ax * v11);
        __half hi, lo;
        split_half(v, hi, lo);
        o[k] = hi;                  // columns [0, 324): hi part
        o[RAFT_CF_LO + k] = lo;     // columns [384, 708): lo part (the conv weights are duplicated over both halves)
    }                               // columns 324..383 / 708..767 stay zero (the buffer is cleared once per call)
}

// Row layout of hx / qx (RAFT_HX = 768 columns, raft_kernels.h): [h_hi 0..127 | h_lo 128..255 | inp_hi 256..383 |
// inp_lo 384..511 | motion_hi 512..637, flow_hi 638..639 | motion_lo 640..765, flow_lo 766..767].
// Every GEMM operand of the update block is carried as a split-fp16 pair (weights duplicated over the hi / lo columns):
// RAFT's 20-step refinement amplifies operand rounding by ~400x on compressed video (DESIGN.md), so single fp16
// operands cannot meet the 1e-3 bar.  The pairs are written by these elementwise kernels or by the GEMM epilogue's
// split-output mode, so the extra precision costs no extra pass over memory -- only a wider K.
//
// context network output (fp32 conv2 output, 256 ch at border-1 geometry): h = tanh(net) -> h32 / hx[0..255],
// inp = relu(inp) -> cols 256..511 of both hx and qx (raft.py:141-143)
__global__ void cnet_split_kernel(const float* __restrict__ cnet, Vol2 vi, __half* __restrict__ hx,
                                  __half* __restrict__ qx, float* __restrict__ h32, Vol2 vo, int ld) {
    const int H = vo.h1 - vo.h0, W = vo.w1 - vo.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(vo.n) * H * W * 256;
    if (idx >= total) return;
    const int c = int(idx % 256);
    const int64_t pos = idx / 256;
    const int xw = int(pos % W), y = int((pos / W) % H), b = int(pos / (int64_t(W) * H));
    const float v = cnet[((int64_t(b) * vi.Hp + y + vi.h0) * vi.Wp + xw + vi.w0) * 256 + c];
    const int64_t orow = (int64_t(b) * vo.Hp + y + vo.h0) * vo.Wp + xw + vo.w0;
    __half hi, lo;
    if (c < 128) {
        const float t = tanhf(v);
        h32[orow * 128 + c] = t;                      // fp32 master copy of the recurrent state
        split_half(t, hi, lo);
        hx[orow * ld + c] = hi;
        hx[orow * ld + 128 + c] = lo;
    } else {
        split_half(fmaxf(v, 0.f), hi, lo);
        hx[orow * ld + 128 + c] = hi;                 // cols 256..383
        hx[orow * ld + 256 + c] = lo;                 // cols 384..511
        qx[orow * ld + 128 + c] = hi;
        qx[orow * ld + 256 + c] = lo;
    }
}

// qx[:, 0:256] = split(r * h) ; qx[:, 512:768] = hx[:, 512:768] (motion features + flow), valid rows.  zr = [z | r].
__global__ void gru_rh_kernel(const __half* __restrict__ hx, const float* __restrict__ h32, const float* __restrict__ zr,
                              __half* __restrict__ qx, Vol2 v, int ld) {
    const int H = v.h1 - v.h0, W = v.w1 - v.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    constexpr int NG = 16 + (RAFT_HX - RAFT_HX_MOTION) / 8;    // 16 groups of 8 for r*h + 32 groups for cols 512..767
    const int64_t total = int64_t(v.n) * H * W * NG;
    if (idx >= total) return;
    const int gidx = int(idx % NG);
    const int64_t pos = idx / NG;
    const int xw = int(pos % W), y = int((pos / W) % H), b = int(pos / (int64_t(W) * H));
    const int64_t row = (int64_t(b) * v.Hp + y + v.h0) * v.Wp + xw + v.w0;
    if (gidx < 16) {
        float hv[8], rv[8];
        *reinterpret_cast<float4*>(hv) = *reinterpret_cast<const float4*>(h32 + row * 128 + gidx * 8);
        *reinterpret_cast<float4*>(hv + 4) = *reinterpret_cast<const float4*>(h32 + row * 128 + gidx * 8 + 4);
        *reinterpret_cast<float4*>(rv) = *reinterpret_cast<const float4*>(zr + row * 256 + 128 + gidx * 8);
        *reinterpret_cast<float4*>(rv + 4) = *reinterpret_cast<const float4*>(zr + row * 256 + 128 + gidx * 8 + 4);
        __align__(16) __half hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) split_half(hv[j] * rv[j], hi[j], lo[j]);
        *reinterpret_cast<uint4*>(qx + row * ld + gidx * 8) = *reinterpret_cast<const uint4*>(hi);
        *reinterpret_cast<uint4*>(qx + row * ld + 128 + gidx * 8) = *reinterpret_cast<const uint4*>(lo);
    } else {
        const int c = RAFT_HX_MOTION + (gidx - 16) * 8;
        *reinterpret_cast<uint4*>(qx + row * ld + c) = *reinterpret_cast<const uint4*>(hx + row * ld + c);
    }
}

// h = (1 - z) * h + z * q   (update.py:55,62) on the fp32 master state; the fp16 copy in hx[:, 0:128] is the GEMM
// operand of the next convolutions.  z and q arrive as fp32 GEMM outputs.
__global__ void gru_update_kernel(__half* __restrict__ hx, float* __restrict__ h32, const float* __restrict__ zr,
                                  const float* __restrict__ q, Vol2 v, int ld) {
    const int H = v.h1 - v.h0, W = v.w1 - v.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * H * W * 16;
    if (idx >= total) return;
    const int g8 = int(idx % 16);
    const int64_t pos = idx / 16;
    const int xw = int(pos % W), y = int((pos / W) % H), b = int(pos / (int64_t(W) * H));
    const int64_t row = (int64_t(b) * v.Hp + y + v.h0) * v.Wp + xw + v.w0;
    float hv[8], zv[8], qv[8];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        *reinterpret_cast<float4*>(hv + 4 * k) = *reinterpret_cast<const float4*>(h32 + row * 128 + g8 * 8 + 4 * k);
        *reinterpret_cast<float4*>(zv + 4 * k) = *reinterpret_cast<const float4*>(zr + row * 256 + g8 * 8 + 4 * k);
        *reinterpret_cast<float4*>(qv + 4 * k) = *reinterpret_cast<const float4*>(q + row * 128 + g8 * 8 + 4 * k);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) hv[j] = (1.f - zv[j]) * hv[j] + zv[j] * qv[j];
#pragma unroll
    for (int k = 0; k < 2; ++k)
        *reinterpret_cast<float4*>(h32 + row * 128 + g8 * 8 + 4 * k) = *reinterpret_cast<const float4*>(hv + 4 * k);
    __align__(16) __half hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) split_half(hv[j], hi[j], lo[j]);
    *reinterpret_cast<uint4*>(hx + row * ld + g8 * 8) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(hx + row * ld + 128 + g8 * 8) = *reinterpret_cast<const uint4*>(lo);
}

// coords1 += delta (fp32, first 2 of 8 GEMM output columns; delta == nullptr initialises coords to the grid);
// flow = coords1 - coords0 written as a split-fp16 pair to the flow slots of hx / qx (hi pair at cols 638..639, lo pair at 766..767) and flow8 (0..3).
__global__ void coords_update_kernel(float* __restrict__ coords1, const float* __restrict__ delta, __half* __restrict__ hx,
                                     __half* __restrict__ qx, __half* __restrict__ flow8, Vol2 v, int ld) {
    const int H = v.h1 - v.h0, W = v.w1 - v.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * H * W;
    if (idx >= total) return;
    const int xw = int(idx % W), y = int((idx / W) % H), b = int(idx / (int64_t(W) * H));
    const int64_t row = (int64_t(b) * v.Hp + y + v.h0) * v.Wp + xw + v.w0;
    float cx, cy;
    if (delta) {
        cx = coords1[idx * 2] + delta[row * 8];
        cy = coords1[idx * 2 + 1] + delta[row * 8 + 1];
    } else {
        cx = float(xw); cy = float(y);
    }
    coords1[idx * 2] = cx;
    coords1[idx * 2 + 1] = cy;
    __half fxh, fxl, fyh, fyl;
    split_half(cx - float(xw), fxh, fxl);
    split_half(cy - float(y), fyh, fyl);
    const uint2 packed = make_uint2(uint32_t(__half_as_ushort(fxh)) | (uint32_t(__half_as_ushort(fyh)) << 16),
                                    uint32_t(__half_as_ushort(fxl)) | (uint32_t(__half_as_ushort(fyl)) << 16));
    *reinterpret_cast<uint32_t*>(hx + row * ld + RAFT_HX_FLOW) = packed.x;                    // (fx_hi, fy_hi)
    *reinterpret_cast<uint32_t*>(hx + row * ld + RAFT_HX_FLOW + RAFT_HX_LO) = packed.y;       // (fx_lo, fy_lo)
    *reinterpret_cast<uint32_t*>(qx + row * ld + RAFT_HX_FLOW) = packed.x;
    *reinterpret_cast<uint32_t*>(qx + row * ld + RAFT_HX_FLOW + RAFT_HX_LO) = packed.y;
    *reinterpret_cast<uint2*>(flow8 + row * 8) = packed;                                      // (fx_hi, fy_hi, fx_lo, fy_lo)
}

// flow slots of hx <- flow8 (the motion conv's 128-wide store has just cleared them)
__global__ void flow_fill_kernel(const __half* __restrict__ flow8, __half* __restrict__ hx, Vol2 v, int ld) {
    const int H = v.h1 - v.h0, W = v.w1 - v.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * H * W;
    if (idx >= total) return;
    const int xw = int(idx % W), y = int((idx / W) % H), b = int(idx / (int64_t(W) * H));
    const int64_t row = (int64_t(b) * v.Hp + y + v.h0) * v.Wp + xw + v.w0;
    const uint2 packed = *reinterpret_cast<const uint2*>(flow8 + row * 8);
    *reinterpret_cast<uint32_t*>(hx + row * ld + RAFT_HX_FLOW) = packed.x;
    *reinterpret_cast<uint32_t*>(hx + row * ld + RAFT_HX_FLOW + RAFT_HX_LO) = packed.y;
}

// RAFT.upsample_flow (raft.py:100-111): convex combination of the 3x3 neighbourhood of 8*flow with
// softmax(mask over the 9 taps); mask channel = k*64 + sy*8 + sx.  mask already carries the 0.25 factor.
// One thread per output pixel pair (both flow components).
// The output is the window [oy, oy+Ho) x [ox, ox+Wo) of the padded flow (InputPadder.unpad, raft.py:41-44).
__global__ void upsample_flow_kernel(const float* __restrict__ coords1, const float* __restrict__ mask, Vol2 v, int n,
                                     int H8, int W8, int oy, int ox, int Ho, int Wo, float* __restrict__ flow_up) {
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(n) * Ho * Wo;
    if (idx >= total) return;
    const int Xo = int(idx % Wo), Yo = int((idx / Wo) % Ho), b = int(idx / (int64_t(Wo) * Ho));
    const int X = Xo + ox, Y = Yo + oy;
    const int x = X >> 3, sx = X & 7, y = Y >> 3, sy = Y & 7;
    const int64_t row = (int64_t(b) * v.Hp + y + v.h0) * v.Wp + x + v.w0;
    const float* m = mask + row * 576 + sy * 8 + sx;
    float mv[9], mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < 9; ++k) { mv[k] = m[k * 64]; mx = fmaxf(mx, mv[k]); }
    float den = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) { mv[k] = __expf(mv[k] - mx); den += mv[k]; }
    float ux = 0.f, uy = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const int yy = y + k / 3 - 1, xx = x + k % 3 - 1;       // F.unfold(3x3, padding=1): zeros outside
        if (yy >= 0 && yy < H8 && xx >= 0 && xx < W8) {
            const int64_t qi = (int64_t(b) * H8 + yy) * W8 + xx;
            ux += mv[k] * 8.f * (coords1[qi * 2] - float(xx));
            uy += mv[k] * 8.f * (coords1[qi * 2 + 1] - float(yy));
        }
    }
    const float inv = 1.f / den;
    flow_up[((int64_t(b) * 2 + 0) * Ho + Yo) * Wo + Xo] = ux * inv;
    flow_up[((int64_t(b) * 2 + 1) * Ho + Yo) * Wo + Xo] = uy * inv;
}

// diagnostics: valid region of channels [c0, c0+cc) of a bordered fp16 volume -> fp32 NCHW
// lo_off > 0: the columns are the hi halves of split pairs whose lo halves sit lo_off columns to the right
__global__ void unpack2d_kernel(const __half* __restrict__ in, Vol2 v, int ld, int c0, int cc, int lo_off,
                                float* __restrict__ out) {
    const int H = v.h1 - v.h0, W = v.w1 - v.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * cc * H * W;
    if (idx >= total) return;
    const int xw = int(idx % W), y = int((idx / W) % H), c = int((idx / (int64_t(W) * H)) % cc);
    const int b = int(idx / (int64_t(W) * H * cc));
    const __half* src = in + ((int64_t(b) * v.Hp + y + v.h0) * v.Wp + xw + v.w0) * ld + c0 + c;
    out[idx] = __half2float(src[0]) + (lo_off > 0 ? __half2float(src[lo_off]) : 0.f);
}

__global__ void unpack2d_f32_kernel(const float* __restrict__ in, Vol2 v, int ld, int c0, int cc, float* __restrict__ out) {
    const int H = v.h1 - v.h0, W = v.w1 - v.w0;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(v.n) * cc * H * W;
    if (idx >= total) return;
    const int xw = int(idx % W), y = int((idx / W) % H), c = int((idx / (int64_t(W) * H)) % cc);
    const int b = int(idx / (int64_t(W) * H * cc));
    out[idx] = in[((int64_t(b) * v.Hp + y + v.h0) * v.Wp + xw + v.w0) * ld + c0 + c];
}

}  // namespace

#define LAUNCH_CHECK() do { VF_CUDA(cudaGetLastError()); return VF_OK; } while (0)

int raft_input_pack(const void* img, int is_u8, int chw, int n, int Hs, int Ws, int pad_top, int pad_left, int H, int W,
                    __half* out, int Hq, int Wq, cudaStream_t s) {
    const int64_t total = int64_t(n) * Hq * Wq;      // rows of 32 channels (16 hi | 16 lo)
    if (is_u8) raft_input_pack_kernel<uint8_t><<<nb(total, 256), 256, 0, s>>>(static_cast<const uint8_t*>(img), n, Hs, Ws, pad_top, pad_left, H, W, chw, out, Hq, Wq);
    else       raft_input_pack_kernel<float><<<nb(total, 256), 256, 0, s>>>(static_cast<const float*>(img), n, Hs, Ws, pad_top, pad_left, H, W, chw, out, Hq, Wq);
    LAUNCH_CHECK();
}
int raft_instnorm_stats(const float* x, const Vol2& v, int C, double* stats, cudaStream_t s) {
    VF_CUDA(cudaMemsetAsync(stats, 0, size_t(v.n) * C * 2 * sizeof(double), s));
    const int H = v.h1 - v.h0;
    if (C > 256) return fail(VF_ERR_INVALID, "instnorm_stats: C=%d > 256", C);
    const int S = 256 / C;       // 4 / 2 / 2 position phases for C = 64 / 96 / 128
    instnorm_stats_kernel<<<dim3(H, v.n), C * S, 0, s>>>(x, v, C, stats);
    LAUNCH_CHECK();
}
int raft_instnorm_apply(const float* a, const double* a_stats, const __half* res_h, const float* res_raw,
                        const double* res_stats, __half* out, const Vol2& v, int C, cudaStream_t s) {
    const int64_t total = int64_t(v.n) * v.Hp * v.Wp * (C / 8);
    instnorm_apply_kernel<<<nb(total, 256), 256, 0, s>>>(a, a_stats, res_h, res_raw, res_stats, out, v, C);
    LAUNCH_CHECK();
}
int raft_add_relu(const __half* a, const __half* b, __half* out, const Vol2& v, int C, cudaStream_t s) {
    const int64_t total = int64_t(v.n) * v.Hp * v.Wp * (C / 8);
    add_relu_kernel<<<nb(total, 256), 256, 0, s>>>(a, b, out, v, C);
    LAUNCH_CHECK();
}
int raft_gather_valid(const __half* in, const Vol2& v, int C, int ld, __half* out, cudaStream_t s) {
    const int64_t total = int64_t(v.n) * (v.h1 - v.h0) * (v.w1 - v.w0) * (C / 8);
    gather_valid_kernel<<<nb(total, 256), 256, 0, s>>>(in, v, C, ld, out);
    LAUNCH_CHECK();
}
int raft_corr_pool(float* corr, int64_t rows, int ld, int off_in, int Hi, int Wi, int off_out, cudaStream_t s) {
    const int64_t total = rows * (Hi / 2) * (Wi / 2);
    if (total <= 0) return VF_OK;
    corr_pool_kernel<<<nb(total, 256), 256, 0, s>>>(corr, rows, ld, off_in, Hi, Wi, off_out);
    LAUNCH_CHECK();
}
int raft_corr_lookup(const float* corr, int ld, const float* coords, int n, int H8, int W8, __half* out, const Vol2& vo,
                     int out_ld, cudaStream_t s) {
    const int64_t warps = int64_t(n) * H8 * W8 * 4;
    corr_lookup_kernel<<<nb(warps * 32, 256), 256, 0, s>>>(corr, ld, coords, n, H8, W8, out, vo, out_ld);
    LAUNCH_CHECK();
}
int raft_corr_operands(const float* f, const Vol2& v, int P8, __half* A, __half* B, cudaStream_t s) {
    const int64_t total = int64_t(v.n) * (v.h1 - v.h0) * (v.w1 - v.w0) * 32;
    corr_operands_kernel<<<nb(total, 256), 256, 0, s>>>(f, v, P8, A, B);
    LAUNCH_CHECK();
}
int raft_cnet_split(const float* cnet, const Vol2& vi, __half* hx, __half* qx, float* h32, const Vol2& vo, int ld,
                    cudaStream_t s) {
    const int64_t total = int64_t(vo.n) * (vo.h1 - vo.h0) * (vo.w1 - vo.w0) * 256;
    cnet_split_kernel<<<nb(total, 256), 256, 0, s>>>(cnet, vi, hx, qx, h32, vo, ld);
    LAUNCH_CHECK();
}
int raft_gru_rh(const __half* hx, const float* h32, const float* zr, __half* qx, const Vol2& v, int ld, cudaStream_t s) {
    const int64_t total = int64_t(v.n) * (v.h1 - v.h0) * (v.w1 - v.w0) * (16 + (RAFT_HX - RAFT_HX_MOTION) / 8);
    gru_rh_kernel<<<nb(total, 256), 256, 0, s>>>(hx, h32, zr, qx, v, ld);
    LAUNCH_CHECK();
}
int raft_gru_update(__half* hx, float* h32, const float* zr, const float* q, const Vol2& v, int ld, cudaStream_t s) {
    const int64_t total = int64_t(v.n) * (v.h1 - v.h0) * (v.w1 - v.w0) * 16;
    gru_update_kernel<<<nb(total, 256), 256, 0, s>>>(hx, h32, zr, q, v, ld);
    LAUNCH_CHECK();
}
int raft_coords_update(float* coords1, const float* delta, __half* hx, __half* qx, __half* flow8, const Vol2& v, int ld,
                       cudaStream_t s) {
    const int64_t total = int64_t(v.n) * (v.h1 - v.h0) * (v.w1 - v.w0);
    coords_update_kernel<<<nb(total, 256), 256, 0, s>>>(coords1, delta, hx, qx, flow8, v, ld);
    LAUNCH_CHECK();
}
int raft_flow_fill(const __half* flow8, __half* hx, const Vol2& v, int ld, cudaStream_t s) {
    const int64_t total = int64_t(v.n) * (v.h1 - v.h0) * (v.w1 - v.w0);
    flow_fill_kernel<<<nb(total, 256), 256, 0, s>>>(flow8, hx, v, ld);
    LAUNCH_CHECK();
}
int raft_upsample_flow(const float* coords1, const float* mask, const Vol2& v, int n, int H8, int W8, int oy, int ox,
                       int Ho, int Wo, float* flow_up, cudaStream_t s) {
    const int64_t total = int64_t(n) * Ho * Wo;
    upsample_flow_kernel<<<nb(total, 256), 256, 0, s>>>(coords1, mask, v, n, H8, W8, oy, ox, Ho, Wo, flow_up);
    LAUNCH_CHECK();
}
int raft_unpack2d_f32(const float* in, const Vol2& v, int ld, int c0, int cc, float* out, cudaStream_t s) {
    const int64_t total = int64_t(v.n) * cc * (v.h1 - v.h0) * (v.w1 - v.w0);
    unpack2d_f32_kernel<<<nb(total, 256), 256, 0, s>>>(in, v, ld, c0, cc, out);
    LAUNCH_CHECK();
}
int raft_unpack2d(const __half* in, const Vol2& v, int ld, int c0, int cc, int lo_off, float* out, cudaStream_t s) {
    const int64_t total = int64_t(v.n) * cc * (v.h1 - v.h0) * (v.w1 - v.w0);
    unpack2d_kernel<<<nb(total, 256), 256, 0, s>>>(in, v, ld, c0, cc, lo_off, out);
    LAUNCH_CHECK();
}

}  // namespace vf
