// torchvision ResNet-18/34/50/101/152 with fc = Identity on the tcgen05 conv-GEMM.
// Replaces `model(batch)` of the ResNet extractor (reference: models/resnet/extract_resnet.py:54-71, 105-110) together
// with its transform (extract_resnet.py:32-38) for the u8 entry.
//
// Layout: channels-last single-fp16 rows of zero-bordered 2-D volumes (conv2d.h).  Every conv is a shifted-row GEMM
// with its BatchNorm folded into the epilogue's scale / bias (and ReLU fused where the block has one); stride-2 convs
// (the 7x7 stem, the 3x3 of a first block, the 1x1 downsample) read a phase repack of their input.  Geometry:
//   stem: phase volume 115x115 (RESNET_STEM_Q) -> output 112x112 at border 2 before / 1 after
//   stage s (0 = stem max pool, 1..4 = layer1..4): H = 56, 56, 28, 14, 7 in a border-1 volume (H+2)^2, kept in its own
//   buffer x[s] so that every stage output can be read back after a forward (vf_resnet_read_stage).
// Precision: fp16 weights and fp16 activations everywhere, fp32 accumulate and epilogue (DESIGN.md §4.6: the CPU
// emulation puts this at <= 5.2e-4 of the 1e-3 bar for every depth).
// Frames are cut into equal chunks of at most max_frames; each chunk size is captured once as a CUDA graph (stem conv
// through layer4) and replayed.
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "conv2d.h"
#include "internal.h"
#include "raft_kernels.h"       // raft_unpack2d (read-back of a bordered fp16 volume)
#include "resnet_kernels.h"

namespace vf {
namespace {

struct Block {
    ConvW c1, c2, c3, down;
    bool has_down = false;
    int stride = 1, cin = 0, planes = 0, cout = 0;
};

Vol2 stage_vol(int n, int H) { return Vol2{n, H + 2, H + 2, 1, H + 1, 1, H + 1}; }
Vol2 stem_vol(int n) { return Vol2{n, RESNET_STEM_Q, RESNET_STEM_Q, 2, 114, 2, 114}; }
const int kStageH[5] = {56, 56, 28, 14, 7};

}  // namespace
}  // namespace vf

using namespace vf;

struct vf_resnet {
    int device = 0, depth = 0, max_frames = 0, dim = 0;
    bool bottleneck = false;
    std::vector<void*> allocs;
    ConvAlloc ca;
    ConvW stem;
    std::vector<Block> blocks[4];
    int stage_c[5] = {64, 0, 0, 0, 0};
    __half *s0 = nullptr, *x[5] = {}, *y = nullptr, *y2 = nullptr, *r = nullptr, *d = nullptr, *ph = nullptr;
    uint8_t *resized = nullptr, *resize_tmp = nullptr;
    size_t resized_cap = 0, tmp_cap = 0;
    int64_t launches = 0;
    cudaStream_t cs = nullptr;
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    bool use_graph = true;
    std::map<int, std::pair<cudaGraphExec_t, int64_t>> graphs;     // chunk size -> (graph, launches in it)
    int last_n = 0;
};

namespace vf {
namespace {

// + 64 KB: the overlapping-row TMA view of a conv input extends (kw-1)*pitch elements past its last row
int ralloc(vf_resnet* h, void** p, size_t bytes) {
    cudaError_t e = cudaMalloc(p, bytes + 65536);
    if (e != cudaSuccess) return fail(VF_ERR_NOMEM, "cudaMalloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
    h->allocs.push_back(*p);
    return VF_OK;
}

int grow(vf_resnet* h, uint8_t** p, size_t* cap, size_t need) {
    if (need <= *cap) return VF_OK;
    if (*p) cudaFree(*p);
    *p = nullptr; *cap = 0;
    VF_CUDA(cudaMalloc(p, need));
    *cap = need;
    return VF_OK;
}

int conv(vf_resnet* h, const ConvW& cw, const __half* X, int pitch, const Vol2& v, __half* out, int ldo, int act,
         cudaStream_t s) {
    h->launches += 1;
    return run_conv(cw, X, pitch, v, out, ldo, 0, act, s);
}

// stem + max pool + layer1..4 on m frames whose stem phase volume is in h->s0; the result is in h->x[4]
int resnet_core(vf_resnet* h, int m, cudaStream_t s) {
    VF_TRY(conv(h, h->stem, h->s0, 16, stem_vol(m), h->y, 64, VF_ACT_RELU, s));
    VF_TRY(resnet_maxpool(h->y, stem_vol(m), 64, h->x[0], stage_vol(m, 56), s));
    h->launches += 1;
    for (int st = 0; st < 4; ++st) {
        const Vol2 vout = stage_vol(m, kStageH[st + 1]);
        for (size_t bi = 0; bi < h->blocks[st].size(); ++bi) {
            const Block& B = h->blocks[st][bi];
            const __half* xin = bi == 0 ? h->x[st] : h->x[st + 1];
            const Vol2 vin = bi == 0 ? stage_vol(m, kStageH[st]) : vout;
            __half* xo = h->x[st + 1];
            if (h->bottleneck) {
                VF_TRY(conv(h, B.c1, xin, B.cin, vin, h->y, B.planes, VF_ACT_RELU, s));
                if (B.stride == 2) {
                    VF_TRY(conv2d_phase_repack(h->y, vin, B.planes, h->ph, vout, s));
                    h->launches += 1;
                    VF_TRY(conv(h, B.c2, h->ph, 4 * B.planes, vout, h->y2, B.planes, VF_ACT_RELU, s));
                } else {
                    VF_TRY(conv(h, B.c2, h->y, B.planes, vout, h->y2, B.planes, VF_ACT_RELU, s));
                }
                VF_TRY(conv(h, B.c3, h->y2, B.planes, vout, h->r, B.cout, VF_ACT_NONE, s));
                if (B.stride == 2) {
                    VF_TRY(conv2d_phase_repack(xin, vin, B.cin, h->ph, vout, s));
                    h->launches += 1;
                }
            } else {
                if (B.stride == 2) {
                    VF_TRY(conv2d_phase_repack(xin, vin, B.cin, h->ph, vout, s));
                    h->launches += 1;
                    VF_TRY(conv(h, B.c1, h->ph, 4 * B.cin, vout, h->y, B.planes, VF_ACT_RELU, s));
                } else {
                    VF_TRY(conv(h, B.c1, xin, B.cin, vout, h->y, B.planes, VF_ACT_RELU, s));
                }
                VF_TRY(conv(h, B.c2, h->y, B.planes, vout, h->r, B.cout, VF_ACT_NONE, s));
            }
            const __half* idn = xin;
            if (B.has_down) {      // stride 2: phase (0,0) of the repacked block input (h->ph)
                VF_TRY(conv(h, B.down, B.stride == 2 ? h->ph : xin, B.stride == 2 ? 4 * B.cin : B.cin, vout, h->d, B.cout,
                            VF_ACT_NONE, s));
                idn = h->d;
            }
            VF_TRY(resnet_add_relu(idn, h->r, xo, vout, B.cout, s));
            h->launches += 1;
        }
    }
    return VF_OK;
}

int prep_network(vf_resnet* h, const TensorTable& T) {
    static const int kBlocks[5][4] = {{2, 2, 2, 2}, {3, 4, 6, 3}, {3, 4, 6, 3}, {3, 4, 23, 3}, {3, 8, 36, 3}};
    const int di = h->depth == 18 ? 0 : h->depth == 34 ? 1 : h->depth == 50 ? 2 : h->depth == 101 ? 3 : 4;
    h->bottleneck = h->depth >= 50;
    const int exp = h->bottleneck ? 4 : 1;
    auto ident = [](int c) { return c; };
    BnFold f;
    auto fold = [&](const std::string& name, int c) -> int {
        if (!bn_fold(T, name, c, &f)) return fail(VF_ERR_INVALID, "resnet_create: missing BatchNorm '%s'", name.c_str());
        return VF_OK;
    };
    // stem: phase rows of 16 channels, 4 (3 used) per phase
    VF_TRY(fold("bn1", 64));
    VF_TRY(prep_stride2_conv(h->ca, h->stem, T, "conv1", 64, 3, 7, 16, 4, -1, 64, &f));
    int cin = 64;
    for (int st = 0; st < 4; ++st) {
        const int planes = 64 << st;
        h->blocks[st].resize(kBlocks[di][st]);
        for (int b = 0; b < kBlocks[di][st]; ++b) {
            Block& B = h->blocks[st][b];
            const std::string p = "layer" + std::to_string(st + 1) + "." + std::to_string(b);
            B.stride = (b == 0 && st > 0) ? 2 : 1;
            B.cin = cin; B.planes = planes; B.cout = planes * exp;
            B.has_down = b == 0 && (B.stride == 2 || cin != B.cout);
            if (h->bottleneck) {
                VF_TRY(fold(p + ".bn1", planes));
                VF_TRY(prep_same_conv(h->ca, B.c1, T, p + ".conv1", planes, cin, 1, 1, cin, ident, planes, &f));
                VF_TRY(fold(p + ".bn2", planes));
                if (B.stride == 2)
                    VF_TRY(prep_stride2_conv(h->ca, B.c2, T, p + ".conv2", planes, planes, 3, 4 * planes, planes, -1, planes, &f));
                else
                    VF_TRY(prep_same_conv(h->ca, B.c2, T, p + ".conv2", planes, planes, 3, 3, planes, ident, planes, &f));
                VF_TRY(fold(p + ".bn3", B.cout));
                VF_TRY(prep_same_conv(h->ca, B.c3, T, p + ".conv3", B.cout, planes, 1, 1, planes, ident, B.cout, &f));
            } else {
                VF_TRY(fold(p + ".bn1", planes));
                if (B.stride == 2)
                    VF_TRY(prep_stride2_conv(h->ca, B.c1, T, p + ".conv1", planes, cin, 3, 4 * cin, cin, -1, planes, &f));
                else
                    VF_TRY(prep_same_conv(h->ca, B.c1, T, p + ".conv1", planes, cin, 3, 3, cin, ident, planes, &f));
                VF_TRY(fold(p + ".bn2", planes));
                VF_TRY(prep_same_conv(h->ca, B.c2, T, p + ".conv2", planes, planes, 3, 3, planes, ident, planes, &f));
            }
            if (B.has_down) {
                VF_TRY(fold(p + ".downsample.1", B.cout));
                if (B.stride == 2)
                    VF_TRY(prep_down_conv(h->ca, B.down, T, p + ".downsample.0", B.cout, cin, B.cout, &f, -1));
                else
                    VF_TRY(prep_same_conv(h->ca, B.down, T, p + ".downsample.0", B.cout, cin, 1, 1, cin, ident, B.cout, &f));
            }
            cin = B.cout;
        }
        h->stage_c[st + 1] = cin;
    }
    h->dim = cin;
    return VF_OK;
}

// fp16 elements per frame of the shared intermediates (y, y2, r, d, ph): the largest any block uses
size_t scratch_per_frame(const vf_resnet* h) {
    size_t e = size_t(stem_vol(1).rows()) * 64;
    for (int st = 0; st < 4; ++st)
        for (const Block& B : h->blocks[st]) {
            const size_t rin = size_t(stage_vol(1, kStageH[B.stride == 2 ? st : st + 1]).rows());
            const size_t rout = size_t(stage_vol(1, kStageH[st + 1]).rows());
            const size_t cand[4] = {rin * B.planes, rout * B.cout, rout * 4 * B.cin, rout * 4 * B.planes};
            for (size_t c : cand) e = c > e ? c : e;
        }
    return e;
}

int balanced_chunk(const vf_resnet* h, int n) {
    const int nchunks = (n + h->max_frames - 1) / h->max_frames;
    return nchunks > 0 ? (n + nchunks - 1) / nchunks : h->max_frames;
}

// the network on m frames (stem phase volume in h->s0) -> out (m x dim fp32), replaying the chunk size's graph
int run_chunk(vf_resnet* h, int m, float* out, cudaStream_t s) {
    if (!h->use_graph || gemm_profile_on()) {
        VF_TRY(resnet_core(h, m, s));
    } else {
        auto it = h->graphs.find(m);
        if (it == h->graphs.end()) {
            const int64_t before = h->launches;
            cudaGraph_t graph = nullptr;
            VF_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed));
            const int st = resnet_core(h, m, s);
            const cudaError_t ce = cudaStreamEndCapture(s, &graph);
            const int64_t n_launch = h->launches - before;
            h->launches = before;
            if (st != VF_OK) { if (graph) cudaGraphDestroy(graph); return st; }
            if (ce != cudaSuccess) return fail(VF_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(ce));
            cudaGraphExec_t exec = nullptr;
            const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ie != cudaSuccess) return fail(VF_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ie));
            // balanced chunks give at most two sizes per call (the chunk and a ragged last chunk): a bounded cache
            // still keeps a long run of varied call sizes from piling up graphs
            if (h->graphs.size() >= 16) {
                cudaGraphExecDestroy(h->graphs.begin()->second.first);
                h->graphs.erase(h->graphs.begin());
            }
            it = h->graphs.emplace(m, std::make_pair(exec, n_launch)).first;
        }
        VF_CUDA(cudaGraphLaunch(it->second.first, s));
        h->launches += it->second.second;
    }
    VF_TRY(resnet_avgpool(h->x[4], stage_vol(m, 7), h->dim, out, s));
    h->launches += 1;
    h->last_n = m;
    return VF_OK;
}

int enter(vf_resnet* h, void* stream) {
    VF_CUDA(cudaSetDevice(h->device));
    VF_CUDA(cudaEventRecord(h->ev_in, static_cast<cudaStream_t>(stream)));
    VF_CUDA(cudaStreamWaitEvent(h->cs, h->ev_in, 0));
    return VF_OK;
}
int leave(vf_resnet* h, void* stream) {
    VF_CUDA(cudaEventRecord(h->ev_out, h->cs));
    VF_CUDA(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), h->ev_out, 0));
    return VF_OK;
}

}  // namespace
}  // namespace vf

extern "C" {

int vf_resnet_create(vf_resnet_t** out, int depth, const vf_named_tensor* tensors, int n_tensors, int device,
                     int max_frames) {
    if (!out || !tensors || n_tensors <= 0) return fail(VF_ERR_INVALID, "resnet_create: null argument");
    *out = nullptr;
    if (depth != 18 && depth != 34 && depth != 50 && depth != 101 && depth != 152)
        return fail(VF_ERR_INVALID, "resnet_create: depth %d is not one of 18, 34, 50, 101, 152", depth);
    if (max_frames < 1) return fail(VF_ERR_INVALID, "resnet_create: max_frames must be >= 1");
    VF_CUDA(cudaSetDevice(device));
    int major = 0;
    VF_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) return fail(VF_ERR_UNSUPPORTED, "device %d is not sm_100; this library is built for sm_100a only", device);
    vf_resnet* h = new vf_resnet();
    h->device = device; h->depth = depth; h->max_frames = max_frames;
    h->ca.wsplit = 1;
    h->ca.alloc = [h](void** p, size_t count, size_t elem) { return ralloc(h, p, count * elem); };
    auto body = [&]() -> int {
        TensorTable T{tensors, n_tensors};
        T.conv_bias = false;                 // torchvision's ResNet convs have no bias
        VF_TRY(prep_network(h, T));
        const size_t F = size_t(max_frames);
        auto alloc_h = [&](__half** p, size_t elems) { return ralloc(h, reinterpret_cast<void**>(p), elems * sizeof(__half)); };
        VF_TRY(alloc_h(&h->s0, F * RESNET_STEM_Q * RESNET_STEM_Q * 16));
        for (int st = 0; st < 5; ++st) VF_TRY(alloc_h(&h->x[st], F * stage_vol(1, kStageH[st]).rows() * h->stage_c[st]));
        const size_t E = F * scratch_per_frame(h);
        VF_TRY(alloc_h(&h->y, E)); VF_TRY(alloc_h(&h->y2, E)); VF_TRY(alloc_h(&h->r, E));
        VF_TRY(alloc_h(&h->d, E)); VF_TRY(alloc_h(&h->ph, E));
        VF_CUDA(cudaStreamCreateWithFlags(&h->cs, cudaStreamNonBlocking));
        VF_CUDA(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
        VF_CUDA(cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming));
        const char* e = getenv("VF_NO_GRAPH");
        h->use_graph = !(e && e[0] == '1');
        return VF_OK;
    };
    const int st = body();
    if (st != VF_OK) { vf_resnet_destroy(h); return st; }
    *out = h;
    return VF_OK;
}

int vf_resnet_destroy(vf_resnet_t* h) {
    if (!h) return VF_OK;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (void* p : h->allocs) cudaFree(p);
    if (h->resized) cudaFree(h->resized);
    if (h->resize_tmp) cudaFree(h->resize_tmp);
    for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);
    if (h->cs) cudaStreamDestroy(h->cs);
    if (h->ev_in) cudaEventDestroy(h->ev_in);
    if (h->ev_out) cudaEventDestroy(h->ev_out);
    delete h;
    return VF_OK;
}

int vf_resnet_feature_dim(const vf_resnet_t* h) { return h ? h->dim : 0; }

int vf_resnet_forward_f32(vf_resnet_t* h, const float* frames, int n, float* out, void* stream) {
    if (!h || !frames || !out) return fail(VF_ERR_INVALID, "resnet_forward_f32: null argument");
    if (n < 0) return fail(VF_ERR_INVALID, "resnet_forward_f32: n = %d", n);
    if (n == 0) return VF_OK;
    VF_TRY(enter(h, stream));
    const int step = balanced_chunk(h, n);
    for (int b0 = 0; b0 < n; b0 += step) {
        const int c = n - b0 < step ? n - b0 : step;
        VF_TRY(resnet_stem_pack_f32(frames + size_t(b0) * 3 * 224 * 224, c, h->s0, h->cs));
        h->launches += 1;
        VF_TRY(run_chunk(h, c, out + size_t(b0) * h->dim, h->cs));
    }
    return leave(h, stream);
}

int vf_resnet_forward_u8(vf_resnet_t* h, const uint8_t* frames, int n, int src_h, int src_w, int swap_rb, float* out,
                         void* stream) {
    if (!h || !frames || !out) return fail(VF_ERR_INVALID, "resnet_forward_u8: null argument");
    if (n < 0 || src_h <= 0 || src_w <= 0) return fail(VF_ERR_INVALID, "resnet_forward_u8: bad shape");
    if (n == 0) return VF_OK;
    // Resize(256): Pillow bilinear, short side to 256 (a pass whose size does not change is skipped, as in Pillow)
    int rh = 0, rw = 0;
    VF_TRY(vf_resize_geometry(src_h, src_w, 256, 1, &rh, &rw));
    const bool resize = rh != src_h || rw != src_w;
    const int cy = center_crop_offset(rh, 224), cx = center_crop_offset(rw, 224);
    VF_TRY(enter(h, stream));
    const int step = balanced_chunk(h, n);
    for (int b0 = 0; b0 < n; b0 += step) {
        const int c = n - b0 < step ? n - b0 : step;
        const uint8_t* src = frames + size_t(b0) * src_h * src_w * 3;
        if (resize) {
            VF_TRY(grow(h, &h->resized, &h->resized_cap, size_t(step) * rh * rw * 3));
            VF_TRY(grow(h, &h->resize_tmp, &h->tmp_cap, size_t(step) * src_h * rw * 3));
            VF_TRY(resize_u8(src, c, src_h, src_w, h->resized, rh, rw, VF_FILTER_BILINEAR, h->resize_tmp, h->cs));
            h->launches += 1;
            src = h->resized;
        }
        VF_TRY(resnet_stem_pack_u8(src, c, rh, rw, cy, cx, swap_rb, h->s0, h->cs));
        h->launches += 1;
        VF_TRY(run_chunk(h, c, out + size_t(b0) * h->dim, h->cs));
    }
    return leave(h, stream);
}

int vf_imagenet_normalize_u8(const uint8_t* src, int n, int src_h, int src_w, int swap_rb, float* dst, void* stream) {
    if (!src || !dst) return fail(VF_ERR_INVALID, "imagenet_normalize: null buffer");
    if (src_h < 224 || src_w < 224) return fail(VF_ERR_INVALID, "imagenet_normalize: %dx%d smaller than the crop", src_h, src_w);
    if (n <= 0) return VF_OK;
    return launch_imagenet_normalize_f32(src, n, src_h, src_w, center_crop_offset(src_h, 224), center_crop_offset(src_w, 224),
                                         swap_rb, dst, static_cast<cudaStream_t>(stream));
}

int vf_resnet_read_stage(vf_resnet_t* h, int stage, float* out, int64_t capacity, int* dims4, void* stream) {
    if (!h || !dims4) return fail(VF_ERR_INVALID, "resnet_read_stage: null argument");
    if (h->last_n <= 0) return fail(VF_ERR_INVALID, "resnet_read_stage: no forward has run");
    if (stage < 0 || stage > 4) return fail(VF_ERR_INVALID, "resnet_read_stage: stage %d outside 0..4", stage);
    const int n = h->last_n, C = h->stage_c[stage], H = kStageH[stage];
    dims4[0] = n; dims4[1] = C; dims4[2] = H; dims4[3] = H;
    if (!out) return VF_OK;
    if (capacity < int64_t(n) * C * H * H) return fail(VF_ERR_INVALID, "resnet_read_stage: capacity too small");
    VF_CUDA(cudaStreamSynchronize(h->cs));      // diagnostics only: the engine stream has finished the last call
    return raft_unpack2d(h->x[stage], stage_vol(n, H), C, 0, C, 0, out, static_cast<cudaStream_t>(stream));
}

int64_t vf_resnet_launch_count(const vf_resnet_t* h) { return h ? h->launches : 0; }

}  // extern "C"
