// RAFT optical flow (full model, 20 refinement iterations) on the tcgen05 conv-GEMM.
// Replaces `RAFT()(image1, image2, iters=20, test_mode=True)` (reference: models/raft/raft_src/raft.py:115-174, called at
// models/raft/extract_raft.py:99 and models/i3d/extract_i3d.py:172) together with InputPadder (raft.py:27-44).
//
// Layout: channels-last fp16 rows of zero-bordered 2-D volumes; every convolution is a shifted-row GEMM
// (conv_gemm_f16): kw taps of one kernel row are one contiguous K run, stride-2 convs run on a space-to-depth
// ("phase") repack of their input, InstanceNorm (fnet) is a stats + apply pass around the raw conv output,
// BatchNorm (cnet, eval) is folded into the conv epilogue.  All-pairs correlation is one 3-term split GEMM per pair
// (fmap1 . fmap2^T / 16, fp32 out) followed by the 3-level average pooling; the per-iteration lookup gathers the
// 4 x 9x9 bilinear windows (the reference's transposed window) straight into the motion encoder's operand rows.
// The GRU operands live in `hx` rows of 768 columns (layout: raft_kernels.h) so that the 1x5 / 5x1 gate convolutions read
// one contiguous run per tap; `qx` is the same row with r*h in place of h.
// Numerics: RAFT's refinement amplifies operand rounding by 2-3 orders of magnitude, so EVERY GEMM operand is a
// split-fp16 pair (activations [hi | lo] with duplicated weight columns, weights as hi + lo passes, W_lo skipped on
// lo-only K blocks): emulated fp32 on the fp16 tensor cores, 1e-5-class agreement with the fp32 reference (DESIGN.md).
// The convex-upsampling mask head and the 8x upsample run once, after the last iteration (the reference evaluates
// them every iteration and discards 19 of the 20 results, raft.py:166-172).
// fnet runs once per frame (the reference encodes every interior frame twice: as image2 of one pair and image1 of
// the next; InstanceNorm is per sample, so the features are identical).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <functional>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "internal.h"
#include "conv2d.h"
#include "raft_kernels.h"

namespace vf {

static const int HX = RAFT_HX;   // hx / qx row layout: raft_kernels.h
static const int CF = RAFT_CF;    // correlation-feature rows: raft_kernels.h

}  // namespace vf

using namespace vf;

struct vf_raft {
    int device = 0, max_frames = 0, max_h = 0, max_w = 0;
    int lead_alloc = 0;         // guard rows in front of every update-block buffer (pointers below are past them)
    std::vector<void*> allocs;
    ConvAlloc ca;               // weight uploads: ralloc into `allocs`; wsplit 2 = weights as hi+lo fp16 pairs
                                // (VF_RAFT_FAST=1: single fp16 weights, outside the parity bar)
    // encoders: [0] = fnet (instance norm), [1] = cnet (batch norm folded)
    struct Enc {
        ConvW conv1, l1[4], l2c1, l2down, l2[3], l3c1, l3down, l3[3], conv2;
    } enc[2];
    ConvW convc1, convc2, convf1, convf2, convm, zr1, q1, zr2, q2, fh1, fh2, mk0, mk2;
    float* sixteenth = nullptr;      // 1/16 for the correlation scale
    // workspace
    __half *s0 = nullptr, *bufA = nullptr, *bufB = nullptr, *bufC = nullptr, *bufD = nullptr, *bufE = nullptr;
    float *fmap32 = nullptr, *cnet32 = nullptr;     // fp32 encoder outputs (border-1 /8 geometry, 256 ch)
    __half *corrA = nullptr, *corrB = nullptr;       // split operands of the correlation GEMM, dense [F][P8][768]
    double *st_a = nullptr, *st_b = nullptr;
    float *corr = nullptr, *coords1 = nullptr, *delta = nullptr, *mask = nullptr;
    float *rawA = nullptr, *rawB = nullptr;     // fp32 conv outputs feeding InstanceNorm
    float *h32 = nullptr, *zr = nullptr, *qb = nullptr;   // fp32 GRU state and gates
    __half *corrfeat = nullptr, *c1 = nullptr, *c2f = nullptr, *f1 = nullptr, *flow8 = nullptr, *hx = nullptr, *qx = nullptr,
           *fh = nullptr, *mk = nullptr;
    int64_t launches = 0;
    // engine-owned stream; everything between the input pack and the convex upsample is replayed as one CUDA graph per
    // (frames, H, W, iterations): ~600-1000 launches and ~1000 tensor-map encodes per window otherwise
    cudaStream_t cs = nullptr;
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    bool use_graph = true;
    std::map<std::tuple<int, int, int, int>, std::pair<cudaGraphExec_t, int64_t>> graphs;
    // geometry of the last call (for debug reads)
    int last_n = 0, last_H8 = 0, last_W8 = 0, corr_ld = 0, P8 = 0;
    Vol2 g8e{}, g8u{};
};

namespace vf {

template <typename Tp>
static int ralloc(vf_raft* h, Tp** p, size_t count) {
    // + 64 KB: the overlapping-row TMA view of a conv input extends (kw-1)*pitch elements past its last row
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(Tp) + 65536);
    if (e != cudaSuccess) return fail(VF_ERR_NOMEM, "cudaMalloc(%zu bytes): %s", count * sizeof(Tp), cudaGetErrorString(e));
    h->allocs.push_back(q);
    *p = static_cast<Tp*>(q);
    return VF_OK;
}

// Both encoders keep their activations as split-fp16 pairs, rows = [hi C | lo C]: the instance-norm encoder's are
// written by the normalisation kernels (fp32 conv outputs), the batch-norm encoder's by the GEMM epilogue's split
// output (norms folded into scale / bias).  The stem reads the split input phase volume.
static int prep_encoder(vf_raft* h, vf_raft::Enc& e, const TensorTable& T, const std::string& p, bool batch, int out_dim) {
    auto ident = [](int c) { return c; };
    BnFold f; const BnFold* bn = nullptr;
    auto fold = [&](const std::string& name, int c) -> int {
        if (!batch) { bn = nullptr; return VF_OK; }
        if (!bn_fold(T, name, c, &f)) return fail(VF_ERR_INVALID, "raft_create: missing BatchNorm '%s'", name.c_str());
        bn = &f; return VF_OK;
    };
    auto same3 = [&](ConvW& cw, const std::string& name, int co, int ci) -> int {
        return prep_same_conv(h->ca, cw, T, name, co, ci, 3, 3, 2 * ci, ident, co, bn, 1.f, [=](int c) { return ci + c; });
    };
    VF_TRY(fold(p + ".norm1", 64));
    // stem: input phase rows = [16 hi | 16 lo], 4 (3 used) channels per phase
    VF_TRY(prep_stride2_conv(h->ca, e.conv1, T, p + ".conv1", 64, 3, 7, 32, 4, 16, 64, bn));
    for (int blk = 0; blk < 2; ++blk)
        for (int cv = 0; cv < 2; ++cv) {
            const std::string b = p + ".layer1." + std::to_string(blk);
            VF_TRY(fold(b + ".norm" + std::to_string(cv + 1), 64));
            VF_TRY(same3(e.l1[blk * 2 + cv], b + ".conv" + std::to_string(cv + 1), 64, 64));
        }
    const int dims[2][2] = {{64, 96}, {96, 128}};
    for (int L = 0; L < 2; ++L) {
        const std::string lp = p + ".layer" + std::to_string(L + 2);
        const int ci = dims[L][0], co = dims[L][1];
        ConvW& c1 = L == 0 ? e.l2c1 : e.l3c1;
        ConvW& dn = L == 0 ? e.l2down : e.l3down;
        ConvW* rest = L == 0 ? e.l2 : e.l3;
        VF_TRY(fold(lp + ".0.norm1", co));
        VF_TRY(prep_stride2_conv(h->ca, c1, T, lp + ".0.conv1", co, ci, 3, 8 * ci, 2 * ci, ci, co, bn));
        VF_TRY(fold(lp + ".0.downsample.1", co));
        VF_TRY(prep_down_conv(h->ca, dn, T, lp + ".0.downsample.0", co, ci, co, bn, ci));
        VF_TRY(fold(lp + ".0.norm2", co));
        VF_TRY(same3(rest[0], lp + ".0.conv2", co, co));
        VF_TRY(fold(lp + ".1.norm1", co));
        VF_TRY(same3(rest[1], lp + ".1.conv1", co, co));
        VF_TRY(fold(lp + ".1.norm2", co));
        VF_TRY(same3(rest[2], lp + ".1.conv2", co, co));
    }
    VF_TRY(prep_same_conv(h->ca, e.conv2, T, p + ".conv2", out_dim, 128, 1, 1, 256, ident, out_dim, nullptr, 1.f,
                          [](int c) { return 128 + c; }));
    return VF_OK;
}

// the shared conv launch (conv2d.h), counted in the handle's launch total
static int run_conv(vf_raft* h, const ConvW& cw, const __half* X, int pitch, const Vol2& v, void* out, int ldo, int out_mode,
                    int act, cudaStream_t s, int split_off = 0, int lead = 0) {
    h->launches += 1;
    return run_conv(cw, X, pitch, v, out, ldo, out_mode, act, s, split_off, lead);
}

// BasicEncoder.forward on m frames whose (split) stem phase volume is in h->s0; the 256-channel output is written in
// fp32 to `out` (border-1 /8 geometry).  Activation rows are split-fp16 pairs of 2C channels in both encoders.
static int run_encoder(vf_raft* h, const vf_raft::Enc& e, bool inst, int m, int H, int W, float* out, int out_dim,
                       cudaStream_t s) {
    const Vol2 g2{m, H / 2 + 3, W / 2 + 3, 2, 2 + H / 2, 2, 2 + W / 2};
    const Vol2 g4{m, H / 4 + 2, W / 4 + 2, 1, 1 + H / 4, 1, 1 + W / 4};
    const Vol2 g8{m, H / 8 + 2, W / 8 + 2, 1, 1 + H / 8, 1, 1 + W / 8};
    __half *x = h->bufA, *y = h->bufB, *r = h->bufC, *r2 = h->bufD, *ph = h->bufE;
    float *rf = h->rawA, *rf2 = h->rawB;
    auto norm_relu = [&](const float* raw, __half* dst, const Vol2& v, int C) -> int {   // dst = split(relu(IN(raw)))
        VF_TRY(raft_instnorm_stats(raw, v, C, h->st_a, s));
        h->launches += 2;
        return raft_instnorm_apply(raw, h->st_a, nullptr, nullptr, nullptr, dst, v, C, s);
    };
    // conv1 + norm1 + relu
    if (inst) { VF_TRY(run_conv(h, e.conv1, h->s0, 32, g2, rf, 64, 1, VF_ACT_NONE, s)); VF_TRY(norm_relu(rf, x, g2, 64)); }
    else      { VF_TRY(run_conv(h, e.conv1, h->s0, 32, g2, x, 128, 2, VF_ACT_RELU, s, 64)); }
    // a stride-1 residual block at geometry v with C channels: x <- relu(x + relu(norm2(conv2(relu(norm1(conv1(x)))))))
    auto res_block = [&](const ConvW& c1, const ConvW& c2, const Vol2& v, int C) -> int {
        if (inst) {
            VF_TRY(run_conv(h, c1, x, 2 * C, v, rf, C, 1, VF_ACT_NONE, s));
            VF_TRY(norm_relu(rf, y, v, C));
            VF_TRY(run_conv(h, c2, y, 2 * C, v, rf, C, 1, VF_ACT_NONE, s));
            VF_TRY(raft_instnorm_stats(rf, v, C, h->st_a, s));
            VF_TRY(raft_instnorm_apply(rf, h->st_a, x, nullptr, nullptr, x, v, C, s));
            h->launches += 2;
        } else {
            VF_TRY(run_conv(h, c1, x, 2 * C, v, y, 2 * C, 2, VF_ACT_RELU, s, C));
            VF_TRY(run_conv(h, c2, y, 2 * C, v, r, 2 * C, 2, VF_ACT_RELU, s, C));
            VF_TRY(raft_add_relu(x, r, x, v, C, s));
            h->launches += 1;
        }
        return VF_OK;
    };
    VF_TRY(res_block(e.l1[0], e.l1[1], g2, 64));
    VF_TRY(res_block(e.l1[2], e.l1[3], g2, 64));
    // a stride-2 residual block: vin (Cin) -> vout (Cout)
    auto down_block = [&](const ConvW& c1, const ConvW& dn, const ConvW& c2, const Vol2& vin, const Vol2& vout, int Cin,
                          int Cout) -> int {
        VF_TRY(conv2d_phase_repack(x, vin, 2 * Cin, ph, vout, s));
        h->launches += 1;
        if (inst) {
            VF_TRY(run_conv(h, c1, ph, 8 * Cin, vout, rf, Cout, 1, VF_ACT_NONE, s));
            VF_TRY(norm_relu(rf, y, vout, Cout));
            VF_TRY(run_conv(h, c2, y, 2 * Cout, vout, rf, Cout, 1, VF_ACT_NONE, s));
            VF_TRY(run_conv(h, dn, ph, 8 * Cin, vout, rf2, Cout, 1, VF_ACT_NONE, s));
            VF_TRY(raft_instnorm_stats(rf, vout, Cout, h->st_a, s));
            VF_TRY(raft_instnorm_stats(rf2, vout, Cout, h->st_b, s));
            VF_TRY(raft_instnorm_apply(rf, h->st_a, nullptr, rf2, h->st_b, x, vout, Cout, s));   // relu(IN(down) + relu(IN(c2)))
            h->launches += 3;
        } else {
            VF_TRY(run_conv(h, c1, ph, 8 * Cin, vout, y, 2 * Cout, 2, VF_ACT_RELU, s, Cout));
            VF_TRY(run_conv(h, c2, y, 2 * Cout, vout, r, 2 * Cout, 2, VF_ACT_RELU, s, Cout));
            VF_TRY(run_conv(h, dn, ph, 8 * Cin, vout, r2, 2 * Cout, 2, VF_ACT_NONE, s, Cout));    // norm3 folded, no relu
            VF_TRY(raft_add_relu(r2, r, x, vout, Cout, s));
            h->launches += 1;
        }
        return VF_OK;
    };
    VF_TRY(down_block(e.l2c1, e.l2down, e.l2[0], g2, g4, 64, 96));
    VF_TRY(res_block(e.l2[1], e.l2[2], g4, 96));
    VF_TRY(down_block(e.l3c1, e.l3down, e.l3[0], g4, g8, 96, 128));
    VF_TRY(res_block(e.l3[1], e.l3[2], g8, 128));
    VF_TRY(run_conv(h, e.conv2, x, 256, g8, out, out_dim, 1, VF_ACT_NONE, s));      // fp32 output
    return VF_OK;
}

}  // namespace vf

extern "C" {

int vf_raft_create(vf_raft_t** out, const vf_named_tensor* tensors, int n_tensors, int device, int max_frames, int max_h,
                   int max_w) {
    if (!out || !tensors || n_tensors <= 0) return fail(VF_ERR_INVALID, "raft_create: null argument");
    *out = nullptr;
    if (max_frames < 2) max_frames = 2;
    if (max_h <= 0 || max_w <= 0) return fail(VF_ERR_INVALID, "raft_create: max frame size required");
    VF_CUDA(cudaSetDevice(device));
    int major = 0;
    VF_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) return fail(VF_ERR_UNSUPPORTED, "device %d is not sm_100; this library is built for sm_100a only", device);
    vf_raft* h = new vf_raft();
    h->device = device; h->max_frames = max_frames;
    h->max_h = (max_h + 7) / 8 * 8; h->max_w = (max_w + 7) / 8 * 8;
    const TensorTable T{tensors, n_tensors};
    auto ident = [](int c) { return c; };
    {
        const char* e = getenv("VF_RAFT_FAST");
        h->ca.wsplit = (e && e[0] == '1') ? 1 : 2;
    }
    h->ca.alloc = [h](void** p, size_t count, size_t elem) { return ralloc(h, reinterpret_cast<char**>(p), count * elem); };
    auto body = [&]() -> int {
        VF_TRY(prep_encoder(h, h->enc[0], T, "fnet", false, 256));
        VF_TRY(prep_encoder(h, h->enc[1], T, "cnet", true, 256));
        const std::string u = "update_block.";
        VF_TRY(prep_same_conv(h->ca, h->convc1, T, u + "encoder.convc1", 256, 324, 1, 1, CF, ident, 256, nullptr, 1.f,
                              [](int c) { return RAFT_CF_LO + c; }));                // lo half of the correlation features
        auto lo256 = [](int c) { return 256 + c; };
        VF_TRY(prep_same_conv(h->ca, h->convc2, T, u + "encoder.convc2", 192, 256, 3, 3, 512, ident, 192, nullptr, 1.f, lo256));
        VF_TRY(prep_same_conv(h->ca, h->convf1, T, u + "encoder.convf1", 128, 2, 7, 7, 8, ident, 128, nullptr, 1.f,
                              [](int c) { return 2 + c; }));                         // flow8 = (fx_hi, fy_hi, fx_lo, fy_lo, ...)
        VF_TRY(prep_same_conv(h->ca, h->convf2, T, u + "encoder.convf2", 64, 128, 3, 3, 256, ident, 64, nullptr, 1.f,
                              [](int c) { return 128 + c; }));
        // reads c2f rows = [cor 192 | flo 64 | cor_lo 192 | flo_lo 64]
        VF_TRY(prep_same_conv(h->ca, h->convm, T, u + "encoder.conv", 126, 256, 3, 3, 512, ident, 128, nullptr, 1.f, lo256));
        // (columns 126, 127 of the motion block hold the flow: raft_flow_fill rewrites them after this conv's 128-wide
        // store.  Clipping the store at 126 columns does not work: a TMA store view whose row is not a multiple of 16 bytes
        // damaged the two neighbouring elements -- measured 5e-3 flow error.)
        // GRU gates read hx / qx rows (layout in raft_kernels.cu): conv input channel c -> column
        //   h (c < 128) -> c [+ lo at 128 + c], inp (128..255) -> 128 + c [+ lo at 256 + c],
        //   motion-out (256..381) and flow (382, 383) -> 256 + c [+ lo at 384 + c]   (12 K blocks, alternately hi / lo)
        auto gmap = [](int c) { return c < 128 ? c : (c < 256 ? 128 + c : 256 + c); };
        auto gmap_lo = [](int c) { return c < 128 ? 128 + c : (c < 256 ? 256 + c : 384 + c); };
        // z and r share their input: one GEMM with N = 256 (z | r)
        for (int dir = 0; dir < 2; ++dir) {
            const std::string sfx = dir == 0 ? "1" : "2";
            const int kh = dir == 0 ? 1 : 5, kw = dir == 0 ? 5 : 1;
            ConvW& zr = dir == 0 ? h->zr1 : h->zr2;
            ConvW& qq = dir == 0 ? h->q1 : h->q2;
            // stack convz | convr weights into one [256, 384, kh, kw] filter
            const float *wz = T.get(u + "gru.convz" + sfx + ".weight", 128 * 384 * 5), *bz = T.get(u + "gru.convz" + sfx + ".bias", 128);
            const float *wr = T.get(u + "gru.convr" + sfx + ".weight", 128 * 384 * 5), *br = T.get(u + "gru.convr" + sfx + ".bias", 128);
            if (!wz || !bz || !wr || !br) return fail(VF_ERR_INVALID, "raft_create: missing GRU gate tensors");
            std::vector<float> wzr(size_t(256) * 384 * 5), bzr(256);
            memcpy(wzr.data(), wz, sizeof(float) * 128 * 384 * 5);
            memcpy(wzr.data() + size_t(128) * 384 * 5, wr, sizeof(float) * 128 * 384 * 5);
            memcpy(bzr.data(), bz, sizeof(float) * 128);
            memcpy(bzr.data() + 128, br, sizeof(float) * 128);
            const vf_named_tensor tmp[2] = {{"zr.weight", wzr.data(), int64_t(wzr.size())}, {"zr.bias", bzr.data(), 256}};
            const TensorTable TT{tmp, 2};
            VF_TRY(prep_same_conv(h->ca, zr, TT, "zr", 256, 384, kh, kw, HX, gmap, 256, nullptr, 1.f, gmap_lo));
            VF_TRY(prep_same_conv(h->ca, qq, T, u + "gru.convq" + sfx, 128, 384, kh, kw, HX, gmap, 128, nullptr, 1.f, gmap_lo));
        }
        VF_TRY(prep_unmerged_conv(h->ca, h->fh1, T, u + "flow_head.conv1", 256, 128, 3, 3, 256, true));    // reads [h_hi | h_lo]
        VF_TRY(prep_same_conv(h->ca, h->fh2, T, u + "flow_head.conv2", 2, 256, 3, 3, 512, ident, 8, nullptr, 1.f, lo256));
        // the convex-upsampling mask is three orders of magnitude less sensitive (4e-6 from fp16 weights): single fp16
        VF_TRY(prep_unmerged_conv(h->ca, h->mk0, T, u + "mask.0", 256, 128, 3, 3, 256, true, 1.f, 1));
        VF_TRY(prep_same_conv(h->ca, h->mk2, T, u + "mask.2", 576, 256, 1, 1, 256, ident, 576, nullptr, 0.25f, nullptr, 1));   // .25 * mask
        {
            const size_t np8 = (size_t(h->max_h / 8) * (h->max_w / 8) + 7) / 8 * 8 + 64;
            std::vector<float> s16(np8, 1.0f / 16.0f);     // corr / sqrt(256) (corr.py:60)
            VF_TRY(ralloc(h, &h->sixteenth, s16.size()));
            VF_CUDA(cudaMemcpy(h->sixteenth, s16.data(), s16.size() * sizeof(float), cudaMemcpyHostToDevice));
        }
        // ---- workspace
        const size_t F = size_t(max_frames), NP = F - 1;
        const int H = h->max_h, W = h->max_w;
        const size_t rows2 = F * (H / 2 + 3) * (W / 2 + 3), rows4 = F * (H / 4 + 2) * (W / 4 + 2);
        const size_t rows8e = F * (H / 8 + 2) * (W / 8 + 2), rows8u = NP * (H / 8 + 6) * (W / 8 + 6);
        const size_t enc_elems = rows2 * 64 > rows4 * 96 ? rows2 * 64 : rows4 * 96;
        VF_TRY(ralloc(h, &h->s0, rows2 * 32));
        VF_TRY(ralloc(h, &h->bufA, 2 * enc_elems)); VF_TRY(ralloc(h, &h->bufB, 2 * enc_elems));   // split rows
        VF_TRY(ralloc(h, &h->bufC, 2 * enc_elems)); VF_TRY(ralloc(h, &h->bufD, 2 * enc_elems));
        VF_TRY(ralloc(h, &h->rawA, enc_elems)); VF_TRY(ralloc(h, &h->rawB, enc_elems));
        const size_t ph_elems = rows4 * 256 > rows8e * 384 ? rows4 * 256 : rows8e * 384;
        VF_TRY(ralloc(h, &h->bufE, 2 * ph_elems));
        VF_TRY(ralloc(h, &h->fmap32, rows8e * 256));
        VF_TRY(ralloc(h, &h->cnet32, rows8e * 256));
        const size_t P = size_t(H / 8) * (W / 8), P8 = (P + 7) / 8 * 8;
        VF_TRY(ralloc(h, &h->corrA, F * P8 * 768));
        VF_TRY(ralloc(h, &h->corrB, F * P8 * 768));
        // rows P .. P8-1 of a frame are never written: they must hold finite values (they only feed unread corr columns)
        VF_CUDA(cudaMemset(h->corrA, 0, F * P8 * 768 * sizeof(__half)));
        VF_CUDA(cudaMemset(h->corrB, 0, F * P8 * 768 * sizeof(__half)));
        VF_TRY(ralloc(h, &h->st_a, F * 128 * 2)); VF_TRY(ralloc(h, &h->st_b, F * 128 * 2));
        const size_t ld = (P8 + P / 4 + P / 16 + P / 64 + 64 + 3) / 4 * 4;
        VF_TRY(ralloc(h, &h->corr, NP * P * ld));
        VF_TRY(ralloc(h, &h->coords1, NP * P * 2));
        // update-block volumes: `lead` zeroed guard rows in front of the first sample (run_conv's row0), see raft_core
        h->lead_alloc = 3 * (W / 8 + 3) + 3;
        auto ualloc = [&](auto** p, size_t ld) -> int {
            const size_t count = (size_t(h->lead_alloc) + rows8u + 8) * ld;
            VF_TRY(ralloc(h, p, count));
            VF_CUDA(cudaMemset(*p, 0, count * sizeof(**p)));
            *p += size_t(h->lead_alloc) * ld;
            return VF_OK;
        };
        VF_TRY(ualloc(&h->corrfeat, CF)); VF_TRY(ualloc(&h->c1, 512));
        VF_TRY(ualloc(&h->c2f, 512));     VF_TRY(ualloc(&h->f1, 256));
        VF_TRY(ualloc(&h->flow8, 8));     VF_TRY(ualloc(&h->hx, HX));
        VF_TRY(ualloc(&h->qx, HX));       VF_TRY(ualloc(&h->zr, 256));
        VF_TRY(ualloc(&h->qb, 128));      VF_TRY(ualloc(&h->fh, 512));
        VF_TRY(ualloc(&h->h32, 128));
        VF_TRY(ualloc(&h->mk, 256));
        VF_TRY(ualloc(&h->delta, 8));     VF_TRY(ualloc(&h->mask, 576));
        VF_CUDA(cudaStreamCreateWithFlags(&h->cs, cudaStreamNonBlocking));
        VF_CUDA(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
        VF_CUDA(cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming));
        {
            const char* e = getenv("VF_NO_GRAPH");
            h->use_graph = !(e && e[0] == '1');
        }
        return VF_OK;
    };
    const int st = body();
    if (st != VF_OK) { vf_raft_destroy(h); return st; }
    *out = h;
    return VF_OK;
}

int vf_raft_destroy(vf_raft_t* h) {
    if (!h) return VF_OK;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (void* p : h->allocs) cudaFree(p);
    for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);
    if (h->cs) cudaStreamDestroy(h->cs);
    if (h->ev_in) cudaEventDestroy(h->ev_in);
    if (h->ev_out) cudaEventDestroy(h->ev_out);
    delete h;
    return VF_OK;
}

}  // extern "C"

namespace vf {

// geometry of the update-block volumes (see raft_core)
static Vol2 update_vol(int NP, int H8, int W8) { return Vol2{NP, H8 + 3, W8 + 3, 0, H8, 0, W8}; }

// encoders -> correlation pyramid -> `iters` refinement steps -> mask head; the stem phase volume is already in h->s0
static int raft_core(vf_raft* h, int F, int H, int W, int iters, cudaStream_t s) {
    const int NP = F - 1, H8 = H / 8, W8 = W / 8, P = H8 * W8, P8 = (P + 7) / 8 * 8;
    VF_TRY(run_encoder(h, h->enc[0], true, F, H, W, h->fmap32, 256, s));
    const Vol2 g8eF{F, H8 + 2, W8 + 2, 1, 1 + H8, 1, 1 + W8};
    VF_TRY(raft_corr_operands(h->fmap32, g8eF, P8, h->corrA, h->corrB, s));
    // ---- all-pairs correlation + pyramid: corr[b] = fmap[b] . fmap[b+1]^T / 16
    int lvl_off[4], lvl_h[4], lvl_w[4];
    lvl_off[0] = 0; lvl_h[0] = H8; lvl_w[0] = W8;
    int ldc = P8;
    for (int l = 1; l < 4; ++l) { lvl_h[l] = lvl_h[l - 1] / 2; lvl_w[l] = lvl_w[l - 1] / 2; lvl_off[l] = ldc; ldc += lvl_h[l] * lvl_w[l]; }
    ldc = (ldc + 3) / 4 * 4;
    for (int b = 0; b < NP; ++b) {
        GemmEpi ep;
        memset(&ep, 0, sizeof(ep));
        ep.out = h->corr + size_t(b) * P * ldc; ep.ldo = ldc; ep.out_f32 = 1; ep.scale = h->sixteenth; ep.act = VF_ACT_NONE;
        // 3-term split product: [f1_hi | f1_lo | f1_hi] . [f2_hi | f2_hi | f2_lo]^T
        VF_TRY(gemm_f16(h->corrA + size_t(b) * P8 * 768, 768, h->corrB + size_t(b + 1) * P8 * 768, 768, P, P8, 768, ep, s));
    }
    for (int l = 1; l < 4; ++l)
        VF_TRY(raft_corr_pool(h->corr, int64_t(NP) * P, ldc, lvl_off[l - 1], lvl_h[l - 1], lvl_w[l - 1], lvl_off[l], s));
    h->launches += NP + 6;
    // ---- context network on frames[:-1] (batch norm folded); reuses s0: the first NP frames' phase rows
    VF_TRY(run_encoder(h, h->enc[1], false, NP, H, W, h->cnet32, 256, s));
    const Vol2 g8e{NP, H8 + 2, W8 + 2, 1, 1 + H8, 1, 1 + W8};
    // update-block volume: 3 zero rows / columns AFTER the valid region only.  In the flattened row space the pad behind
    // image row y is also the pad in front of row y+1, and the pad below sample b the pad above sample b+1; in front of
    // the first sample sit `lead` zeroed guard rows (a merged-kw tap starts kw/2 rows early, so they must be real rows,
    // not TMA out-of-bounds fill).  (H8+3)(W8+3) rows per sample instead of (H8+6)(W8+6): 12 % fewer GEMM rows at 270x480.
    const Vol2 g8u = update_vol(NP, H8, W8);
    const int lead = 3 * g8u.Wp + 3;
    const size_t rows8u = size_t(g8u.rows());
    // zero the update-block operand buffers once: their border rows are read as conv padding
    VF_CUDA(cudaMemsetAsync(h->hx, 0, rows8u * HX * sizeof(__half), s));
    VF_CUDA(cudaMemsetAsync(h->qx, 0, rows8u * HX * sizeof(__half), s));
    VF_CUDA(cudaMemsetAsync(h->flow8, 0, rows8u * 8 * sizeof(__half), s));
    VF_CUDA(cudaMemsetAsync(h->corrfeat, 0, rows8u * CF * sizeof(__half), s));
    VF_TRY(raft_cnet_split(h->cnet32, g8e, h->hx, h->qx, h->h32, g8u, HX, s));
    VF_TRY(raft_coords_update(h->coords1, nullptr, h->hx, h->qx, h->flow8, g8u, HX, s));    // coords1 = grid, flow = 0
    h->launches += 4;
    for (int it = 0; it < iters; ++it) {
        VF_TRY(raft_corr_lookup(h->corr, ldc, h->coords1, NP, H8, W8, h->corrfeat, g8u, CF, s));
        // every intermediate is a split pair written by the GEMM epilogue: rows = [hi | lo]
        VF_TRY(run_conv(h, h->convc1, h->corrfeat, CF, g8u, h->c1, 512, 2, VF_ACT_RELU, s, 256, lead));
        VF_TRY(run_conv(h, h->convc2, h->c1, 512, g8u, h->c2f, 512, 2, VF_ACT_RELU, s, 256, lead));         // cols 0..191 | 256..447
        VF_TRY(run_conv(h, h->convf1, h->flow8, 8, g8u, h->f1, 256, 2, VF_ACT_RELU, s, 128, lead));
        VF_TRY(run_conv(h, h->convf2, h->f1, 256, g8u, h->c2f + 192, 512, 2, VF_ACT_RELU, s, 256, lead));   // cols 192..255 | 448..511
        VF_TRY(run_conv(h, h->convm, h->c2f, 512, g8u, h->hx + RAFT_HX_MOTION, HX, 2, VF_ACT_RELU, s, RAFT_HX_LO, lead));   // 512..637 | 640..765
        VF_TRY(raft_flow_fill(h->flow8, h->hx, g8u, HX, s));
        h->launches += 1;
        for (int dir = 0; dir < 2; ++dir) {
            const ConvW& zr = dir == 0 ? h->zr1 : h->zr2;
            const ConvW& qq = dir == 0 ? h->q1 : h->q2;
            VF_TRY(run_conv(h, zr, h->hx, HX, g8u, h->zr, 256, 1, VF_ACT_SIGMOID, s, 0, lead));
            VF_TRY(raft_gru_rh(h->hx, h->h32, h->zr, h->qx, g8u, HX, s));
            VF_TRY(run_conv(h, qq, h->qx, HX, g8u, h->qb, 128, 1, VF_ACT_TANH, s, 0, lead));
            VF_TRY(raft_gru_update(h->hx, h->h32, h->zr, h->qb, g8u, HX, s));
        }
        VF_TRY(run_conv(h, h->fh1, h->hx, HX, g8u, h->fh, 512, 2, VF_ACT_RELU, s, 256, lead));
        VF_TRY(run_conv(h, h->fh2, h->fh, 512, g8u, h->delta, 8, 1, VF_ACT_NONE, s, 0, lead));
        VF_TRY(raft_coords_update(h->coords1, h->delta, h->hx, h->qx, h->flow8, g8u, HX, s));
        h->launches += 6;
    }
    // ---- mask head (once, after the last iteration)
    VF_TRY(run_conv(h, h->mk0, h->hx, HX, g8u, h->mk, 256, 0, VF_ACT_RELU, s, 0, lead));
    VF_TRY(run_conv(h, h->mk2, h->mk, 256, g8u, h->mask, 576, 1, VF_ACT_NONE, s, 0, lead));
    h->last_n = NP; h->last_H8 = H8; h->last_W8 = W8; h->corr_ld = ldc; h->P8 = P8; h->g8e = g8e; h->g8u = g8u;
    return VF_OK;
}

}  // namespace vf

extern "C" {

int vf_raft_flow(vf_raft_t* h, const void* frames, int is_u8, int chw_layout, int n_frames, int Hs, int Ws, int iters,
                 int unpad, float* out, void* stream) {
    if (!h || !frames || !out) return fail(VF_ERR_INVALID, "raft_flow: null argument");
    if (n_frames < 2 || n_frames > h->max_frames) return fail(VF_ERR_INVALID, "raft_flow: %d frames outside [2, %d]", n_frames, h->max_frames);
    if (iters < 1) return fail(VF_ERR_INVALID, "raft_flow: iters must be >= 1");
    // InputPadder 'sintel' (raft.py:29-34)
    const int pad_h = (((Hs / 8) + 1) * 8 - Hs) % 8, pad_w = (((Ws / 8) + 1) * 8 - Ws) % 8;
    const int pl = pad_w / 2, pt = pad_h / 2;
    const int H = Hs + pad_h, W = Ws + pad_w;
    if (H > h->max_h || W > h->max_w || H < 16 || W < 16)
        return fail(VF_ERR_INVALID, "raft_flow: padded frame %dx%d outside the workspace (%dx%d)", H, W, h->max_h, h->max_w);
    const int F = n_frames, NP = F - 1, H8 = H / 8, W8 = W / 8, P = H8 * W8;
    cudaStream_t user = static_cast<cudaStream_t>(stream), s = h->cs;
    VF_CUDA(cudaSetDevice(h->device));
    VF_CUDA(cudaEventRecord(h->ev_in, user));
    VF_CUDA(cudaStreamWaitEvent(s, h->ev_in, 0));
    VF_TRY(raft_input_pack(frames, is_u8, chw_layout, F, Hs, Ws, pt, pl, H, W, h->s0, H / 2 + 3, W / 2 + 3, s));
    h->launches += 1;
    if (!h->use_graph || gemm_profile_on()) {
        VF_TRY(raft_core(h, F, H, W, iters, s));
    } else {
        auto key = std::make_tuple(F, H, W, iters);
        auto it = h->graphs.find(key);
        if (it == h->graphs.end()) {
            const int64_t before = h->launches;
            cudaGraph_t graph = nullptr;
            VF_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed));
            const int st = raft_core(h, F, H, W, iters, s);
            const cudaError_t ce = cudaStreamEndCapture(s, &graph);
            const int64_t n_launch = h->launches - before;
            h->launches = before;
            if (st != VF_OK) { if (graph) cudaGraphDestroy(graph); return st; }
            if (ce != cudaSuccess) return fail(VF_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(ce));
            cudaGraphExec_t exec = nullptr;
            const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ie != cudaSuccess) return fail(VF_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ie));
            // bounded cache: a list of videos of many resolutions (or ragged last calls) must not pile up executable
            // graphs; an evicted graph that is still running is freed by the runtime when it completes
            if (h->graphs.size() >= 16) {
                cudaGraphExecDestroy(h->graphs.begin()->second.first);
                h->graphs.erase(h->graphs.begin());
            }
            it = h->graphs.emplace(key, std::make_pair(exec, n_launch)).first;
        }
        VF_CUDA(cudaGraphLaunch(it->second.first, s));
        h->launches += it->second.second;
        // geometry bookkeeping normally done inside raft_core
        h->last_n = NP; h->last_H8 = H8; h->last_W8 = W8;
        {
            int ldc = (P + 7) / 8 * 8, lh = H8, lw = W8;
            for (int l = 1; l < 4; ++l) { lh /= 2; lw /= 2; ldc += lh * lw; }
            h->corr_ld = (ldc + 3) / 4 * 4;
        }
        h->g8e = Vol2{NP, H8 + 2, W8 + 2, 1, 1 + H8, 1, 1 + W8};
        h->g8u = update_vol(NP, H8, W8);
    }
    // ---- convex upsampling, once
    if (unpad) VF_TRY(raft_upsample_flow(h->coords1, h->mask, h->g8u, NP, H8, W8, pt, pl, Hs, Ws, out, s));
    else       VF_TRY(raft_upsample_flow(h->coords1, h->mask, h->g8u, NP, H8, W8, 0, 0, H, W, out, s));
    h->launches += 1;
    VF_CUDA(cudaEventRecord(h->ev_out, s));
    VF_CUDA(cudaStreamWaitEvent(user, h->ev_out, 0));
    return VF_OK;
}

int vf_raft_padded_size(int Hs, int Ws, int* H, int* W) {
    if (!H || !W || Hs <= 0 || Ws <= 0) return fail(VF_ERR_INVALID, "raft_padded_size: bad argument");
    *H = Hs + (((Hs / 8) + 1) * 8 - Hs) % 8;
    *W = Ws + (((Ws / 8) + 1) * 8 - Ws) % 8;
    return VF_OK;
}

int vf_raft_debug_read(vf_raft_t* h, int what, float* out, int64_t capacity, int* dims4, void* stream) {
    if (!h || !dims4 || h->last_n <= 0) return fail(VF_ERR_INVALID, "raft_debug_read: no forward has run");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    VF_CUDA(cudaStreamSynchronize(h->cs));      // diagnostics only: the engine stream has finished the last call
    const int n = h->last_n, H8 = h->last_H8, W8 = h->last_W8;
    int64_t need = 0;
    if (what == 0) { dims4[0] = n + 1; dims4[1] = 256; dims4[2] = H8; dims4[3] = W8; }
    else if (what == 1) { dims4[0] = n; dims4[1] = 256; dims4[2] = H8; dims4[3] = W8; }
    else if (what == 2) { dims4[0] = n; dims4[1] = 128; dims4[2] = H8; dims4[3] = W8; }
    else if (what == 3) { dims4[0] = n; dims4[1] = 2; dims4[2] = H8; dims4[3] = W8; }
    else if (what == 4) { dims4[0] = n; dims4[1] = 324; dims4[2] = H8; dims4[3] = W8; }
    else if (what == 5) { dims4[0] = n; dims4[1] = H8 * W8; dims4[2] = 1; dims4[3] = h->corr_ld; }   // raw pyramid rows
    else return fail(VF_ERR_INVALID, "raft_debug_read: unknown tensor id %d", what);
    need = int64_t(dims4[0]) * dims4[1] * dims4[2] * dims4[3];
    if (!out) return VF_OK;
    if (capacity < need) return fail(VF_ERR_INVALID, "raft_debug_read: capacity too small");
    if (what == 5) {
        VF_CUDA(cudaMemcpyAsync(out, h->corr, size_t(need) * sizeof(float), cudaMemcpyDeviceToDevice, s));
        return VF_OK;
    }
    if (what == 0) { Vol2 v = h->g8e; v.n = n + 1; return raft_unpack2d_f32(h->fmap32, v, 256, 0, 256, out, s); }
    if (what == 1) return raft_unpack2d_f32(h->cnet32, h->g8e, 256, 0, 256, out, s);
    if (what == 2) return raft_unpack2d(h->hx, h->g8u, HX, 0, 128, 128, out, s);                     // GRU hidden state (hi + lo)
    if (what == 3) return raft_unpack2d(h->hx, h->g8u, HX, RAFT_HX_FLOW, 2, RAFT_HX_LO, out, s);     // low-res flow (hi + lo)
    return raft_unpack2d(h->corrfeat, h->g8u, CF, 0, 324, RAFT_CF_LO, out, s);                               // last lookup (hi + lo)
}

int64_t vf_raft_launch_count(const vf_raft_t* h) { return h ? h->launches : 0; }

}  // extern "C"
