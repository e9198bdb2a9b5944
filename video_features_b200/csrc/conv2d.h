// 2-D convolution layer on the tcgen05 shifted-row conv GEMM, shared by the RAFT encoders (raft.cu) and ResNet
// (resnet.cu): filter re-layout + BatchNorm folding at create time, the conv launch, and the space-to-depth ("phase")
// repack that lets a stride-2 conv run as a stride-1 shifted-row GEMM.
//
// Activations are channels-last fp16 rows of zero-bordered 2-D volumes [n][Hp][Wp][C] (Vol2).  Every convolution is
// conv_gemm_f16: the kw taps of one kernel row are one contiguous K run of kw*pitch elements; a stride-2 conv reads
// the phase repack of its input, where phase (ph, pw) of output position q holds input position 2(q-B)+(ph,pw).
#pragma once
#include <stdint.h>

#include <functional>
#include <string>
#include <vector>

#include "internal.h"

namespace vf {

// zero-bordered 2-D volume [n][Hp][Wp][C]; valid region [h0,h1) x [w0,w1)
struct Vol2 {
    int n, Hp, Wp, h0, h1, w0, w1;
    int64_t rows() const { return int64_t(n) * Hp * Wp; }
    int H() const { return h1 - h0; }
    int W() const { return w1 - w0; }
};

struct ConvW {       // a convolution prepared for conv_gemm_f16
    int n_out = 0;          // GEMM N (padded to a multiple of 8)
    int ntaps = 0, k_per_tap = 0;
    std::vector<int> dh, dw0;   // per tap: row offset (in kernel rows) and the column shift of its first element
    int nsplit = 1;             // 2: w = [hi (ntaps*k_per_tap) | lo (same)] along K (ConvGeom::nsplit)
    unsigned long long lo_mask = 0;   // K blocks (per tap) holding only lo-half activation columns (ConvGeom::lo_mask)
    __half* w = nullptr;
    float *scale = nullptr, *bias = nullptr;
};

// Where a network's device weights go, and how they are stored.  alloc(p, count, elem_bytes) allocates count
// elements on the device (owned and freed by the network); wsplit is the default weight precision: 1 single fp16,
// 2 hi + lo fp16 pairs.
struct ConvAlloc {
    std::function<int(void**, size_t, size_t)> alloc;
    int wsplit = 1;
    template <typename Tp>
    int operator()(Tp** p, size_t count) const {
        void* q = nullptr;
        VF_TRY(alloc(&q, count, sizeof(Tp)));
        *p = static_cast<Tp*>(q);
        return VF_OK;
    }
};

// name -> host fp32 tensor of the expected element count (null when missing or mis-shaped).  conv_bias: the
// network's convolutions carry a bias tensor ("<conv>.bias"); false (torchvision ResNet) reads none.
struct TensorTable {
    const vf_named_tensor* t; int n;
    bool conv_bias = true;
    const float* get(const std::string& name, int64_t numel) const {
        for (int i = 0; i < n; ++i)
            if (name == t[i].name) return t[i].numel == numel ? t[i].data : nullptr;
        return nullptr;
    }
};

// eval-mode BatchNorm (eps 1e-5) as a per-channel scale / shift applied after the conv
struct BnFold { std::vector<float> scale, shift; };
bool bn_fold(const TensorTable& T, const std::string& p, int c, BnFold* f);

// Generic filter re-layout.  w: [co][ci][kh][kw]; col(dh, dw, c) -> K column or -1.  Output rows padded to n_out.
// col_lo (optional): a second K column receiving the same weight -- the column of the operand's lo half when the
// activation is stored as a split-fp16 pair.  b (optional): conv bias.
int upload_conv(const ConvAlloc& A, ConvW& cw, const float* w, const float* b, int co, int ci, int kh, int kw, int n_out,
                int Ktot, const std::function<int(int, int, int)>& col, const float* bn_scale, const float* bn_shift,
                float extra_scale, const std::function<int(int, int, int)>& col_lo = nullptr, int nsplit = -1);

// stride-1 kh x kw conv whose input rows have `pitch` channels with the conv's channel c stored at column chan(c):
// taps = kernel rows, each a run of kw*pitch elements starting (kw/2) positions to the left.
int prep_same_conv(const ConvAlloc& A, ConvW& cw, const TensorTable& T, const std::string& name, int co, int ci, int kh,
                   int kw, int pitch, const std::function<int(int)>& chan, int n_out, const BnFold* bn,
                   float extra_scale = 1.f, const std::function<int(int)>& chan_lo = nullptr, int nsplit = -1);
// same, but every (kh, kw) position is its own tap reading `ci` channels at column offset 0 of rows with a wider pitch
// (dup: the operand row holds [x_hi (ci) | x_lo (ci)], the weight is written to both halves)
int prep_unmerged_conv(const ConvAlloc& A, ConvW& cw, const TensorTable& T, const std::string& name, int co, int ci, int kh,
                       int kw, int n_out, bool dup, float extra_scale = 1.f, int nsplit = -1);
// stride-2 k x k conv (pad k/2) on the phase repack of its input: phase volume row q holds x[2(q-B)+p] with B =
// border-before (2 for k=7, 1 for k=3); filter index = 2a + p - 1 for tap a (k=7: a in 0..3, k=3: a in 0..1).
// Row layout: `pitch` channels per position, channel c of phase (ph,pw) at (ph*2+pw)*phase_stride + c, and -- when the
// activation is a split-fp16 pair -- its lo half `lo_off` columns further (lo_off < 0: single fp16).
int prep_stride2_conv(const ConvAlloc& A, ConvW& cw, const TensorTable& T, const std::string& name, int co, int ci, int k,
                      int pitch, int phase_stride, int lo_off, int n_out, const BnFold* bn);
// 1x1 stride-2 downsample: phase (0,0) of the repacked row = its first ci channels, followed (lo_off = ci) by their
// lo halves when the activation is a split-fp16 pair (lo_off < 0: single fp16)
int prep_down_conv(const ConvAlloc& A, ConvW& cw, const TensorTable& T, const std::string& name, int co, int ci, int n_out,
                   const BnFold* bn, int lo_off);

// out_mode: 0 fp16, 1 fp32, 2 split-fp16 pair (hi at column n, lo at column split_off + n of the same rows)
// lead: guard rows in front of X and out (both pointers are past them); the GEMM covers them and writes them as zeros
int run_conv(const ConvW& cw, const __half* X, int pitch, const Vol2& v, void* out, int ldo, int out_mode, int act,
             cudaStream_t s, int split_off = 0, int lead = 0);

// space-to-depth for a stride-2 3x3 (pad 1) or 1x1 consumer: out[q][(ph*2+pw)*C + c] = in_valid[2(q-1)+ph][2(q'-1)+pw][c]
// (zero outside the valid region); out is a border-1 volume at half resolution with 4*C channels.
int conv2d_phase_repack(const __half* in, const Vol2& vi, int C, __half* out, const Vol2& vo, cudaStream_t s);

}  // namespace vf
