/* libvfeat.so -- C ABI of the B200-native video-feature engine.
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes, returns an int status
 * (VF_OK == 0) and never throws.  Device buffers are raw CUDA device pointers owned by the
 * caller; `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Handles
 * are opaque, own their device weights + workspace, and are not shared between threads.
 *
 * Each function names the reference interface it replaces
 * (Kamino666/video_features @ dc9df59e, paths relative to the reference root).
 */
#ifndef VFEAT_H_
#define VFEAT_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VF_OK 0
#define VF_ERR_INVALID 1   /* bad argument */
#define VF_ERR_CUDA 2      /* a CUDA runtime / driver call failed */
#define VF_ERR_NOMEM 3
#define VF_ERR_UNSUPPORTED 4

#define VF_ACT_NONE 0
#define VF_ACT_QUICKGELU 1 /* x * sigmoid(1.702 x) */
#define VF_ACT_RELU 2
#define VF_ACT_SIGMOID 3
#define VF_ACT_TANH 4

#define VF_FILTER_BILINEAR 2 /* PIL.Image.BILINEAR */
#define VF_FILTER_BICUBIC 3  /* PIL.Image.BICUBIC  */

/* ABI version; bumped on any signature change. */
int vf_version(void);
/* Text of the last error raised on the calling thread ("" if none). */
const char* vf_last_error(void);

/* ---- sampler: utils/utils.py:297-333 `extract_frames` index arithmetic -------------------------
 * method "uni": n = param; "fix": n = (int)(frame_cnt / fps * param).  Writes
 * np.linspace(1, frame_cnt-2, n).astype(int) into out_idx (capacity cap) and n into *out_n;
 * out_idx == NULL only queries n. */
int vf_sample_indices(const char* method, int param, int64_t frame_cnt, double fps, int64_t* out_idx, int64_t cap,
                      int64_t* out_n);
/* contiguous chunk shard of `n_items` over `n_parts` as torch.chunk does (main.py:49-53):
 * part p gets [*begin, *end); parts beyond the last non-empty chunk get begin == end. */
int vf_shard_range(int64_t n_items, int n_parts, int part, int64_t* begin, int64_t* end);

/* ---- PIL-compatible resample: Pillow Image.resize as used by torchvision Resize in the CLIP
 * transform (models/CLIP/extract_clip.py:112) and models/i3d/transforms/transforms.py:121,125.
 * src: n frames HWC uint8 (3 channels) on the device; dst: n x out_h x out_w x 3 uint8.
 * tmp: device scratch of n*in_h*out_w*3 bytes (horizontal pass output); byte-exact with Pillow. */
int vf_resize_u8(const uint8_t* src, int n, int in_h, int in_w, uint8_t* dst, int out_h, int out_w, int filter,
                 uint8_t* tmp, void* stream);
/* output geometry of "short side -> size" (torchvision Resize(int) / ResizeImproved). */
int vf_resize_geometry(int in_h, int in_w, int size, int to_smaller_edge, int* out_h, int* out_w);

/* ---- CLIP transform: ToTensor + Normalize + CenterCrop(224) (clip.clip._transform as invoked at
 * models/CLIP/extract_clip.py:107-113,125-126).  src: n x src_h x src_w x 3 uint8 (already
 * resized); dst: n x 3 x 224 x 224 fp32, bit-exact with torchvision's fp32 arithmetic. */
int vf_clip_normalize_u8(const uint8_t* src, int n, int src_h, int src_w, float* dst, void* stream);

/* ---- tensor-core GEMM (exported for the parity tests): D = act(A . B^T * scale + bias)
 * A: M x K fp16 (row pitch lda elements), B: N x K fp16 (torch Linear weight layout),
 * D: fp16 or fp32 (out_f32, row pitch ldd elements, 16-byte aligned rows), bias/scale: fp32 [N] or NULL. */
int vf_gemm_f16(const void* A, int lda, const void* B, int ldb, int M, int N, int K, void* D, int ldd, int out_f32,
                const float* bias, const float* scale, int act, void* stream);
/* D += act(A . B^T * scale + bias), D fp32: the add happens in the L2 (TMA reduction), each element exactly once -- the
 * residual-stream update `x = x + attn(...)` / `x = x + mlp(...)` of clip/model.py ResidualAttentionBlock.forward. */
int vf_gemm_f16_accumulate(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* D, int ldd,
                           const float* bias, const float* scale, int act, void* stream);
/* Same GEMM with the result written as a split-fp16 pair: D[m][n] = fp16(v) and D[m][split_off + n] = fp16(v - fp16(v))
 * (split_off >= N, multiple of 8, ldd >= split_off + N).  RAFT's GEMM -> GEMM activations are carried this way: the
 * consumer's weights are duplicated over both halves, which restores ~22 mantissa bits on the activation operand. */
int vf_gemm_f16_split(const void* A, int lda, const void* B, int ldb, int M, int N, int K, void* D, int ldd, int split_off,
                      const float* bias, const float* scale, int act, void* stream);

/* Roofline instrumentation (bench.py): while enabled on the calling thread, every tcgen05 GEMM launch of any handle
 * is bracketed by CUDA events on its stream.  _read synchronises the device and returns the summed device time (ms),
 * the launch count and the EXECUTED flops (2*M*N*K including zero-padded K blocks and hi/lo weight passes). */
int vf_gemm_profile(int enable);
int vf_gemm_profile_read(double* ms, int64_t* launches, double* executed_flops);

/* ---- CLIP ViT-B/32 image tower: replaces `clip.load(...)` + `model.encode_image(frames)`
 * (models/CLIP/extract_clip.py:47,128).  Weight pointers are HOST fp32 arrays in openai layout. */
typedef struct vf_clip_layer_weights {
    const float *ln_1_w, *ln_1_b;           /* [768] */
    const float *in_proj_w, *in_proj_b;     /* [2304,768], [2304] */
    const float *out_proj_w, *out_proj_b;   /* [768,768], [768] */
    const float *ln_2_w, *ln_2_b;           /* [768] */
    const float *c_fc_w, *c_fc_b;           /* [3072,768], [3072] */
    const float *c_proj_w, *c_proj_b;       /* [768,3072], [768] */
} vf_clip_layer_weights;

typedef struct vf_clip_weights {
    const float* conv1_w;                   /* [768,3,32,32] */
    const float* class_embedding;           /* [768] */
    const float* positional_embedding;      /* [50,768] */
    const float *ln_pre_w, *ln_pre_b, *ln_post_w, *ln_post_b; /* [768] */
    const float* proj;                      /* [768,512] */
    vf_clip_layer_weights layers[12];
} vf_clip_weights;

typedef struct vf_clip vf_clip_t;

/* Uploads weights to `device` (fp16 GEMM operands, fp32 vectors) and allocates workspace for
 * chunks of `chunk_frames` frames (0 = default). */
int vf_clip_create(vf_clip_t** out, const vf_clip_weights* w, int device, int chunk_frames);
/* Same for the reference's other ViT-B feature type: patch_size 32 ('CLIP-ViT-B/32', identical to vf_clip_create) or 16
 * ('CLIP-ViT-B/16': conv1_w is [768,3,16,16], positional_embedding [197,768]; same width, depth, heads and output size).
 * Reference: models/CLIP/extract_clip.py:42-47 (clip.load(feature_type) for either name). */
int vf_clip_create_vit(vf_clip_t** out, const vf_clip_weights* w, int device, int chunk_frames, int patch_size);
int vf_clip_destroy(vf_clip_t* h);
/* encode_image on n already-transformed frames: frames n x 3 x 224 x 224 fp32 (device) -> out n x 512 fp32. */
int vf_clip_encode_f32(vf_clip_t* h, const float* frames, int n, float* out, void* stream);
/* Fused transform + encode_image: frames n x src_h x src_w x 3 uint8 (device, as the decoder delivers
 * them, channel order untouched) -> Resize(224,bicubic) -> CenterCrop(224) -> normalise -> tower. */
int vf_clip_encode_u8(vf_clip_t* h, const uint8_t* frames, int n, int src_h, int src_w, float* out, void* stream);
/* Same with HOST buffers: stages H2D copies of the frames and the D2H copy of the features on
 * `stream` and synchronises it before returning (the call ExtractCLIP.extract makes per video). */
int vf_clip_encode_u8_host(vf_clip_t* h, const uint8_t* frames_host, int n, int src_h, int src_w, float* out_host,
                           void* stream);
/* Host frames in, features left ON THE DEVICE in out_dev (n x 512 fp32, ordered on `stream`) -- what a rank hands to the
 * all-gather of main.py's --device_ids dispatch (main.py:49-53) -- and, when out_host is not NULL, copied to the host as
 * well.  Returns once the host frames have been consumed (and out_host, if given, is complete). */
int vf_clip_encode_u8_host_dev(vf_clip_t* h, const uint8_t* frames_host, int n, int src_h, int src_w, float* out_dev,
                               float* out_host, void* stream);

/* Asynchronous form of the two calls above: returns once the copies and kernels are enqueued.  `frames_host` and `out_host`
 * must be pinned and stay untouched until vf_clip_wait(h, *ticket) returns; out_dev (may be NULL) is ordered on `stream`
 * like any other device output.  Calls in flight share the handle's staging slots under event ordering, so the H2D copy
 * of call k+1 overlaps the tower of call k -- the pattern of a list of videos (reference: the per-video loop of
 * models/CLIP/extract_clip.py:70-88, where nothing overlaps).  At most 4 calls are in flight; a fifth blocks on the
 * oldest.  One enqueuing host thread per handle; vf_clip_wait may be called from another thread. */
int vf_clip_encode_u8_host_async(vf_clip_t* h, const uint8_t* frames_host, int n, int src_h, int src_w, float* out_dev,
                                 float* out_host, void* stream, int64_t* ticket);
int vf_clip_wait(vf_clip_t* h, int64_t ticket);
/* Diagnostics / parity tests: the attention half of resblock `layer` alone -- x: n_frames*50 x 768 fp16 (the ln_1 output),
 * out: n_frames*50 x 768 fp16 = concat_heads(softmax(q k^T / 8) v) BEFORE the out-projection (third-party clip
 * ResidualAttentionBlock.attention / nn.MultiheadAttention).  fused = 1: the QKV-projection + attention kernel the tower
 * runs; fused = 0: QKV GEMM, then the stand-alone attention kernel. */
int vf_clip_block_attention(vf_clip_t* h, int layer, const void* x, int n_frames, void* out, int fused, void* stream);
/* number of kernels this library has launched on behalf of `h` so far (diagnostics / bench). */
int64_t vf_clip_launch_count(const vf_clip_t* h);
/* Roofline instrumentation for bench.py: while enabled, every tensor-core GEMM launch of `h` is bracketed by a
 * pair of CUDA events recorded on the launching stream.  vf_clip_profile_read synchronises the device, returns the
 * summed GEMM device time (ms), the number of GEMM launches and their algorithmic FLOPs (2*M*N*K), and resets. */
int vf_clip_profile(vf_clip_t* h, int enable);
int vf_clip_profile_read(vf_clip_t* h, double* gemm_ms, int64_t* gemm_launches, double* gemm_flops);
/* device ms per kernel category of the last vf_clip_profile_read window: [0] GEMM, [1] LayerNorm, [2] attention,
 * [3] frame transform (resize / normalise / patchify). */
int vf_clip_profile_categories(const vf_clip_t* h, double* ms4);

/* ---- I3D (Inception-3D) feature extractor: replaces `I3D(400, modality)(x, features=True)`
 * (models/i3d/i3d_src/i3d_net.py:238-264, called at models/i3d/extract_i3d.py:186).
 * One conv unit = Conv3d (no bias) + BatchNorm3d (eval) + ReLU (Unit3Dpy, i3d_net.py:37-105); weights are HOST fp32
 * in the checkpoint's own layout.  Unit order: conv3d_1a_7x7, conv3d_2b_1x1, conv3d_2c_3x3, then for each of
 * mixed_3b,3c,4b,4c,4d,4e,4f,5b,5c: branch_0, branch_1.0, branch_1.1, branch_2.0, branch_2.1, branch_3.1. */
#define VF_I3D_UNITS 57
typedef struct vf_conv_unit {
    const float* w;                               /* [cout, cin, k, k, k] */
    const float *bn_w, *bn_b, *bn_mean, *bn_var;  /* [cout] */
    int cout, cin, k;
} vf_conv_unit;
typedef struct vf_i3d_weights {
    vf_conv_unit units[VF_I3D_UNITS];
} vf_i3d_weights;
typedef struct vf_i3d vf_i3d_t;

/* in_channels: 3 (rgb stream) or 2 (flow stream).  Workspace is sized for max_stacks clips of max_T frames. */
int vf_i3d_create(vf_i3d_t** out, const vf_i3d_weights* w, int in_channels, int device, int max_stacks, int max_T);
int vf_i3d_destroy(vf_i3d_t* h);
/* clips: n x C x T x 224 x 224 fp32 on the device (the tensor the reference passes to I3D) -> out n x 1024 fp32. */
int vf_i3d_forward_f32(vf_i3d_t* h, const float* clips, int n, int T, float* out, void* stream);
/* rgb stream with the T2 transform fused (extract_i3d.py:62-66): frames n x T x Hr x Wr x 3 uint8 on the device,
 * already resized (vf_resize_u8, bilinear, short side 256) -> TensorCenterCrop(224) -> 2x/255-1 -> I3D. */
int vf_i3d_forward_u8(vf_i3d_t* h, const uint8_t* frames, int n, int T, int Hr, int Wr, float* out, void* stream);
/* same, stack b = frames [b * stack_stride, b * stack_stride + T) of the buffer (stack_stride >= T, in frames): the rgb
 * stream of the reference is `stack[:-1]` of the 65-frame stacks the flow stream also reads (extract_i3d.py:150-158). */
int vf_i3d_forward_u8_strided(vf_i3d_t* h, const uint8_t* frames, int n, int T, int64_t stack_stride, int Hr, int Wr,
                              float* out, void* stream);
/* flow stream with the T3 transform fused (extract_i3d.py:67-73): flow n x T x 2 x H x W fp32 on the device (the RAFT
 * output, still padded) -> crop 224 -> clamp(+-20) -> 128+255/40 f -> round -> 2x/255-1 -> I3D. */
int vf_i3d_forward_flow(vf_i3d_t* h, const float* flow, int n, int T, int H, int W, float* out, void* stream);
/* Diagnostics: copy a retained internal activation (0: conv3d_1a, 1: conv3d_2c, 3: mixed_5b, 4: mixed_5c) of the
 * last forward to fp32 NCTHW; dims5 receives (n, C, T, H, W); out == NULL only queries the shape. */
int vf_i3d_read_stage(vf_i3d_t* h, int stage, float* out, int64_t capacity, int* dims5, void* stream);
int64_t vf_i3d_launch_count(const vf_i3d_t* h);

/* ---- RAFT optical flow: replaces `RAFT()(image1, image2, iters=20, test_mode=True)` + InputPadder
 * (models/raft/raft_src/raft.py:27-44,115-174; called at models/raft/extract_raft.py:94-104 and
 * models/i3d/extract_i3d.py:172).  Weights: the checkpoint's tensors by name (keys of raft-sintel.pth without the
 * "module." prefix), HOST fp32. */
typedef struct vf_named_tensor {
    const char* name;
    const float* data;
    int64_t numel;
} vf_named_tensor;
typedef struct vf_raft vf_raft_t;

/* Workspace is sized for windows of max_frames frames of at most max_h x max_w pixels (before /8 padding). */
int vf_raft_create(vf_raft_t** out, const vf_named_tensor* tensors, int n_tensors, int device, int max_frames, int max_h,
                   int max_w);
int vf_raft_destroy(vf_raft_t* h);
/* Flow between consecutive frames of a window: frames n_frames x (Hs x Ws x 3 if !chw_layout else 3 x Hs x Ws), uint8
 * or fp32 in [0,255] on the device, RGB order as given; == model(pad(frames)[:-1], pad(frames)[1:]).
 * out: (n_frames-1) x 2 x Ho x Wo fp32 with (Ho,Wo) = (Hs,Ws) if unpad (extract_raft.py:101) else the /8-padded size
 * (extract_i3d.py:172 never unpads; query it with vf_raft_padded_size). */
int vf_raft_flow(vf_raft_t* h, const void* frames, int is_u8, int chw_layout, int n_frames, int Hs, int Ws, int iters,
                 int unpad, float* out, void* stream);
int vf_raft_padded_size(int Hs, int Ws, int* H, int* W);
/* Diagnostics: internal tensors of the last call as fp32 NCHW at 1/8 resolution.  what: 0 fnet features (all
 * frames), 1 cnet output (raw), 2 GRU hidden state, 3 low-res flow, 4 last correlation lookup (324 ch),
 * 5 the correlation pyramid rows (n, H8*W8, 1, row pitch): level l at cumulative offset of the level sizes. */
int vf_raft_debug_read(vf_raft_t* h, int what, float* out, int64_t capacity, int* dims4, void* stream);
int64_t vf_raft_launch_count(const vf_raft_t* h);

/* ---- ResNet-18/34/50/101/152 frame features: replaces `model(batch)` with
 * model = torchvision.models.resnet{depth}(pretrained=True), eval, fc = Identity (models/resnet/extract_resnet.py:54-71,
 * called at :109).  Weights: torchvision's state_dict tensors by name ("conv1.weight", "layer1.0.bn1.running_var", ...),
 * HOST fp32; num_batches_tracked and fc.* are not read. */
typedef struct vf_resnet vf_resnet_t;
/* Workspace for max_frames frames per chunk; a call with more frames runs in equal chunks. */
int vf_resnet_create(vf_resnet_t** out, int depth, const vf_named_tensor* tensors, int n_tensors, int device, int max_frames);
int vf_resnet_destroy(vf_resnet_t* h);
/* 512 (depth 18, 34) or 2048 (50, 101, 152) */
int vf_resnet_feature_dim(const vf_resnet_t* h);
/* frames: n x 3 x 224 x 224 fp32 on the device, normalised (extract_resnet.py:106-109 `model(batch)`);
 * out: n x feature_dim fp32 on the device. */
int vf_resnet_forward_f32(vf_resnet_t* h, const float* frames, int n, float* out, void* stream);
/* frames: n x src_h x src_w x 3 uint8 on the device -> Resize(256, Pillow bilinear) -> CenterCrop(224) -> ToTensor ->
 * Normalize(ImageNet) -> net (extract_resnet.py:32-38 then :109); swap_rb: the frames are BGR (cv2) and are read as
 * RGB (extract_resnet.py:142). */
int vf_resnet_forward_u8(vf_resnet_t* h, const uint8_t* frames, int n, int src_h, int src_w, int swap_rb, float* out,
                         void* stream);
/* CenterCrop(224) -> ToTensor -> Normalize(ImageNet mean / std) of n resized uint8 HWC frames (extract_resnet.py:35-37)
 * -> n x 3 x 224 x 224 fp32 on the device; swap_rb as above. */
int vf_imagenet_normalize_u8(const uint8_t* src, int n, int src_h, int src_w, int swap_rb, float* dst, void* stream);
/* Diagnostics: a stage output of the last chunk of the last call as fp32 NCHW; stage 0 = stem + max pool (64 x 56 x
 * 56), 1..4 = layer1..4.  out = NULL only fills dims4. */
int vf_resnet_read_stage(vf_resnet_t* h, int stage, float* out, int64_t capacity, int* dims4, void* stream);
int64_t vf_resnet_launch_count(const vf_resnet_t* h);

#ifdef __cplusplus
}
#endif
#endif /* VFEAT_H_ */
