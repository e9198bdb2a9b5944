// 2-D convolution layer shared by RAFT and ResNet (declarations and layout notes: conv2d.h).
#include <math.h>
#include <string.h>

#include "common.cuh"
#include "conv2d.h"

namespace vf {

int upload_conv(const ConvAlloc& A, ConvW& cw, const float* w, const float* b, int co, int ci, int kh, int kw, int n_out,
                int Ktot, const std::function<int(int, int, int)>& col, const float* bn_scale, const float* bn_shift,
                float extra_scale, const std::function<int(int, int, int)>& col_lo, int nsplit) {
    if (nsplit < 0) nsplit = A.wsplit;
    cw.nsplit = nsplit;
    const size_t Kall = size_t(Ktot) * nsplit;
    std::vector<__half> B(size_t(n_out) * Kall, __float2half_rn(0.f));
    std::vector<char> has_hi(size_t(Ktot), 0);      // K columns that multiply a hi (or single-fp16) activation
    for (int o = 0; o < co; ++o)
        for (int c = 0; c < ci; ++c)
            for (int a = 0; a < kh; ++a)
                for (int d = 0; d < kw; ++d) {
                    const int k = col(a, d, c);
                    if (k < 0) continue;
                    if (k >= Ktot) return fail(VF_ERR_INVALID, "conv upload: filter column out of range");
                    const float wf = w[((size_t(o) * ci + c) * kh + a) * kw + d];
                    const __half wv = __float2half_rn(wf);
                    const __half wl = __float2half_rn(wf - __half2float(wv));
                    B[size_t(o) * Kall + k] = wv;
                    has_hi[k] = 1;
                    if (nsplit == 2) B[size_t(o) * Kall + Ktot + k] = wl;
                    if (col_lo) {
                        const int k2 = col_lo(a, d, c);
                        if (k2 >= Ktot) return fail(VF_ERR_INVALID, "conv upload: filter column out of range");
                        if (k2 >= 0) {
                            B[size_t(o) * Kall + k2] = wv;
                            if (nsplit == 2) B[size_t(o) * Kall + Ktot + k2] = wl;
                        }
                    }
                }
    std::vector<float> sc(n_out, 0.f), bi(n_out, 0.f);
    for (int o = 0; o < co; ++o) {
        const float s = (bn_scale ? bn_scale[o] : 1.f) * extra_scale;
        sc[o] = s;
        bi[o] = (b ? b[o] : 0.f) * s + (bn_shift ? bn_shift[o] : 0.f) * extra_scale;
    }
    cw.n_out = n_out;
    // a K block none of whose columns meets a hi half needs only the W_hi pass (a_lo . w_lo < 2^-22 of the product)
    cw.lo_mask = 0;
    const int kpt_blocks = (cw.k_per_tap + 63) / 64;
    if (nsplit == 2 && kpt_blocks <= 64 && cw.ntaps * cw.k_per_tap == Ktot) {
        unsigned long long m = ~0ull;
        for (int t = 0; t < cw.ntaps; ++t)
            for (int kk = 0; kk < kpt_blocks; ++kk) {
                bool any_hi = false;
                for (int j = kk * 64; j < (kk + 1) * 64 && j < cw.k_per_tap; ++j) any_hi |= has_hi[size_t(t) * cw.k_per_tap + j] != 0;
                if (any_hi) m &= ~(1ull << kk);
            }
        cw.lo_mask = kpt_blocks == 64 ? m : (m & ((1ull << kpt_blocks) - 1));
    }
    VF_TRY(A(&cw.w, B.size()));
    VF_TRY(A(&cw.scale, size_t(n_out)));
    VF_TRY(A(&cw.bias, size_t(n_out)));
    VF_CUDA(cudaMemcpy(cw.w, B.data(), B.size() * sizeof(__half), cudaMemcpyHostToDevice));
    VF_CUDA(cudaMemcpy(cw.scale, sc.data(), n_out * sizeof(float), cudaMemcpyHostToDevice));
    VF_CUDA(cudaMemcpy(cw.bias, bi.data(), n_out * sizeof(float), cudaMemcpyHostToDevice));
    return VF_OK;
}

bool bn_fold(const TensorTable& T, const std::string& p, int c, BnFold* f) {
    const float *g = T.get(p + ".weight", c), *b = T.get(p + ".bias", c), *m = T.get(p + ".running_mean", c),
                *v = T.get(p + ".running_var", c);
    if (!g || !b || !m || !v) return false;
    f->scale.resize(c); f->shift.resize(c);
    for (int i = 0; i < c; ++i) {
        const float s = g[i] / sqrtf(v[i] + 1e-5f);
        f->scale[i] = s;
        f->shift[i] = b[i] - m[i] * s;
    }
    return true;
}

// the conv's weight and (when the table's convolutions carry one) bias
static int conv_tensors(const TensorTable& T, const std::string& name, int64_t wnumel, int co, const float** w,
                        const float** b) {
    *w = T.get(name + ".weight", wnumel);
    *b = T.conv_bias ? T.get(name + ".bias", co) : nullptr;
    if (!*w || (T.conv_bias && !*b)) return fail(VF_ERR_INVALID, "create: missing or mis-shaped tensor '%s'", name.c_str());
    return VF_OK;
}

int prep_same_conv(const ConvAlloc& A, ConvW& cw, const TensorTable& T, const std::string& name, int co, int ci, int kh,
                   int kw, int pitch, const std::function<int(int)>& chan, int n_out, const BnFold* bn,
                   float extra_scale, const std::function<int(int)>& chan_lo, int nsplit) {
    const float *w, *b;
    VF_TRY(conv_tensors(T, name, int64_t(co) * ci * kh * kw, co, &w, &b));
    cw.ntaps = kh; cw.k_per_tap = kw * pitch;
    cw.dh.clear(); cw.dw0.clear();
    for (int a = 0; a < kh; ++a) { cw.dh.push_back(a - kh / 2); cw.dw0.push_back(-(kw / 2)); }
    const int kpt = cw.k_per_tap;
    return upload_conv(A, cw, w, b, co, ci, kh, kw, n_out, kh * kpt,
                       [=](int a, int d, int c) { return a * kpt + d * pitch + chan(c); },
                       bn ? bn->scale.data() : nullptr, bn ? bn->shift.data() : nullptr, extra_scale,
                       chan_lo ? std::function<int(int, int, int)>([=](int a, int d, int c) {
                           const int k = chan_lo(c);
                           return k < 0 ? -1 : a * kpt + d * pitch + k;
                       }) : nullptr, nsplit);
}

int prep_unmerged_conv(const ConvAlloc& A, ConvW& cw, const TensorTable& T, const std::string& name, int co, int ci, int kh,
                       int kw, int n_out, bool dup, float extra_scale, int nsplit) {
    const float *w, *b;
    VF_TRY(conv_tensors(T, name, int64_t(co) * ci * kh * kw, co, &w, &b));
    const int kpt = dup ? 2 * ci : ci;
    cw.ntaps = kh * kw; cw.k_per_tap = kpt;
    cw.dh.clear(); cw.dw0.clear();
    for (int a = 0; a < kh; ++a)
        for (int d = 0; d < kw; ++d) { cw.dh.push_back(a - kh / 2); cw.dw0.push_back(d - kw / 2); }
    return upload_conv(A, cw, w, b, co, ci, kh, kw, n_out, kh * kw * kpt,
                       [=](int a, int d, int c) { return (a * kw + d) * kpt + c; }, nullptr, nullptr, extra_scale,
                       dup ? std::function<int(int, int, int)>([=](int a, int d, int c) { return (a * kw + d) * kpt + ci + c; })
                           : nullptr, nsplit);
}

int prep_stride2_conv(const ConvAlloc& A, ConvW& cw, const TensorTable& T, const std::string& name, int co, int ci, int k,
                      int pitch, int phase_stride, int lo_off, int n_out, const BnFold* bn) {
    const float *w, *b;
    VF_TRY(conv_tensors(T, name, int64_t(co) * ci * k * k, co, &w, &b));
    const int na = (k == 7) ? 4 : 2, before = (k == 7) ? 2 : 1;
    cw.ntaps = na; cw.k_per_tap = na * pitch;
    cw.dh.clear(); cw.dw0.clear();
    for (int a = 0; a < na; ++a) { cw.dh.push_back(a - before); cw.dw0.push_back(-before); }
    const int kpt = cw.k_per_tap;
    // invert (kh, kw) -> (a, ph), (bq, pw): kh = 2a + ph - 1
    auto col = [=](int kh, int kw, int c) {
        const int a = (kh + 1) / 2, ph = (kh + 1) % 2, bq = (kw + 1) / 2, pw = (kw + 1) % 2;
        return a * kpt + bq * pitch + (ph * 2 + pw) * phase_stride + c;
    };
    return upload_conv(A, cw, w, b, co, ci, k, k, n_out, na * kpt, col,
                       bn ? bn->scale.data() : nullptr, bn ? bn->shift.data() : nullptr, 1.f,
                       lo_off >= 0 ? std::function<int(int, int, int)>([=](int kh, int kw, int c) { return col(kh, kw, c) + lo_off; })
                                   : nullptr);
}

int prep_down_conv(const ConvAlloc& A, ConvW& cw, const TensorTable& T, const std::string& name, int co, int ci, int n_out,
                   const BnFold* bn, int lo_off) {
    const float *w, *b;
    VF_TRY(conv_tensors(T, name, int64_t(co) * ci, co, &w, &b));
    cw.ntaps = 1; cw.k_per_tap = lo_off >= 0 ? lo_off + ci : ci;
    cw.dh = {0}; cw.dw0 = {0};
    return upload_conv(A, cw, w, b, co, ci, 1, 1, n_out, cw.k_per_tap, [=](int, int, int c) { return c; },
                       bn ? bn->scale.data() : nullptr, bn ? bn->shift.data() : nullptr, 1.f,
                       lo_off >= 0 ? std::function<int(int, int, int)>([=](int, int, int c) { return lo_off + c; }) : nullptr);
}

int run_conv(const ConvW& cw, const __half* X, int pitch, const Vol2& v, void* out, int ldo, int out_mode, int act,
             cudaStream_t s, int split_off, int lead) {
    ConvGeom g;
    memset(&g, 0, sizeof(g));
    g.ntaps = cw.ntaps; g.k_per_tap = cw.k_per_tap; g.nsplit = cw.nsplit; g.lo_mask = cw.lo_mask;
    for (int j = 0; j < cw.ntaps; ++j) g.tap_off[j] = cw.dh[j] * v.Wp + cw.dw0[j];
    g.mask = 1; g.row0 = lead;
    g.Tp = 1; g.Hp = v.Hp; g.Wp = v.Wp; g.t0 = 0; g.t1 = 1; g.h0 = v.h0; g.h1 = v.h1; g.w0 = v.w0; g.w1 = v.w1;
    X -= size_t(lead) * pitch;
    out = static_cast<char*>(out) - size_t(lead) * ldo * (out_mode == 1 ? 4 : 2);
    GemmEpi ep;
    memset(&ep, 0, sizeof(ep));
    ep.out = out; ep.ldo = ldo; ep.out_f32 = out_mode == 1; ep.bias = cw.bias; ep.scale = cw.scale; ep.act = act;
    ep.split_off = out_mode == 2 ? split_off : 0;
    return conv_gemm_f16(X, pitch, v.rows() + lead, cw.w, cw.n_out, g, ep, s);
}

namespace {

__global__ void phase_repack_kernel(const __half* __restrict__ in, Vol2 vi, int C, __half* __restrict__ out, Vol2 vo) {
    const int cg = C >> 3;
    const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t total = int64_t(vo.n) * vo.Hp * vo.Wp * 4 * cg;
    if (idx >= total) return;
    const int c8 = int(idx % cg);
    const int p = int((idx / cg) % 4);
    const int64_t pos = idx / (4 * cg);
    const int wq = int(pos % vo.Wp), hq = int((pos / vo.Wp) % vo.Hp), b = int(pos / (int64_t(vo.Wp) * vo.Hp));
    const int y = 2 * (hq - 1) + (p >> 1), x = 2 * (wq - 1) + (p & 1);     // valid-region coordinates of the input
    uint4 v = make_uint4(0, 0, 0, 0);
    if (y >= 0 && y < vi.h1 - vi.h0 && x >= 0 && x < vi.w1 - vi.w0)
        v = __ldg(reinterpret_cast<const uint4*>(in + ((int64_t(b) * vi.Hp + y + vi.h0) * vi.Wp + x + vi.w0) * C + c8 * 8));
    *reinterpret_cast<uint4*>(out + pos * (4 * C) + p * C + c8 * 8) = v;
}

}  // namespace

int conv2d_phase_repack(const __half* in, const Vol2& vi, int C, __half* out, const Vol2& vo, cudaStream_t s) {
    const int64_t total = int64_t(vo.n) * vo.Hp * vo.Wp * 4 * (C / 8);
    phase_repack_kernel<<<unsigned((total + 255) / 256), 256, 0, s>>>(in, vi, C, out, vo);
    VF_CUDA(cudaGetLastError());
    return VF_OK;
}

}  // namespace vf
