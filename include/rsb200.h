/*
 * rsb200.h -- C ABI of librsb200.so: the B200 (sm_100a) kernels behind RoboSat's segmentation hot path.
 *
 * The reference (mapbox/robosat @ cbb1c73) has no FFI of its own: its "operator interface" for this
 * path is a handful of PyTorch call sites. Every entry point below names the reference call site it
 * replaces (file:line under /root/reference). Host code (robosat_b200/*.py) binds these with ctypes.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless the name ends in _host
 *   - the library never allocates or frees user tensors and never synchronises: all work is enqueued
 *     on the `stream` argument (a cudaStream_t passed as void*)
 *   - return value: 0 on success, negative RSB_E_* on failure; rsb_last_error() gives the message
 *     (thread local). There is NO CPU fallback: without a usable sm_100 device every compute entry fails.
 *   - activations are NHWC fp16 ("channels last"), accumulators fp32; weights are pre-packed fp16
 *   - two precisions: "fast" (one fp16 plane per tensor) and "strict" (hi + lo fp16 planes, see rsb_conv_desc.split)
 */
#ifndef RSB200_H
#define RSB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSB_OK 0
#define RSB_E_INVALID -1   /* bad argument / unsupported shape */
#define RSB_E_CUDA -2      /* CUDA runtime or driver error */
#define RSB_E_NODEVICE -3  /* no sm_100 device / driver entry point missing */
#define RSB_E_UNSUPPORTED -4 /* (host codecs only) valid input of a kind this entry point does not handle: use another decoder */

#define RSB_MAX_SEGS 16
#define RSB_MAX_SRCS 4

int rsb_version(void);
/* sizeof(rsb_conv_src), sizeof(rsb_conv_seg), sizeof(rsb_conv_desc), sizeof(rsb_rowconv_desc) as compiled into the library,
 * so that a binding (ctypes, cgo, ...) can verify its struct declarations before the first call */
void rsb_abi_layout(int32_t* out4);
const char* rsb_last_error(void);
/* 0 if a compute-capability-10.x device is current and the TMA driver entry point resolves */
int rsb_device_ok(void);

/* ---------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution on tcgen05 tensor cores (fp16 x fp16 -> fp32 in tensor memory).
 *
 * Replaces every nn.Conv2d (+ folded eval BatchNorm, + ReLU, + residual add, + nearest x2 upsample,
 * + channel concat) the forward pass runs:
 *   resnet conv1 / layer1-4 Bottleneck convs      robosat/unet.py:122-130 (torchvision resnet.py Bottleneck.forward)
 *   ConvRelu.forward                              robosat/unet.py:44
 *   DecoderBlock.forward (interpolate + ConvRelu) robosat/unet.py:73
 *   torch.cat([enc, dec], dim=1)                  robosat/unet.py:134-137
 *   final 1x1 conv + bias                         robosat/unet.py:141
 *
 * One output tile = 128 "tile-space" pixels (box TW x TH x TN of one source view) x BLOCK_N output
 * channels. The contraction is a list of segments; each segment is one TMA box load per 64-channel
 * block from source view `src` displaced by (dh, dw) pixels, multiplied by the next 64 columns of the
 * packed weight matrix [phases*Cout][K]. Strided convs use parity views of the input, the nearest
 * x2 upsample uses 4 output phases of 2x2 taps on the low-resolution input (pre-summed weights),
 * channel concat uses two sources; none of them materialises an intermediate tensor.
 */
typedef struct rsb_conv_src {
    const void* ptr;      /* fp16 base of the view (already offset for parity / padding) */
    int64_t pitch_w;      /* element strides of the view */
    int64_t pitch_h;
    int64_t pitch_n;
    int32_t C;            /* innermost extent (channels, or window elements for overlapped views) */
    int32_t W, H, N;      /* extents of the view (TMA zero-fills outside) */
    int64_t plane;        /* split precision only: element stride from the hi plane (ptr) to the lo plane of the same view */
} rsb_conv_src;

typedef struct rsb_conv_seg {
    int32_t src;          /* index into srcs[] */
    int32_t dh, dw;       /* displacement in tile-space pixels, for phase (0,0) */
    int32_t cblocks;      /* number of 64-element blocks taken from that source */
} rsb_conv_seg;

typedef struct rsb_conv_desc {
    int32_t nsrc;
    rsb_conv_src srcs[RSB_MAX_SRCS];
    int32_t nseg;
    rsb_conv_seg segs[RSB_MAX_SEGS];

    const void* weights;  /* fp16 [phases * Cout][K], K = 64 * sum(cblocks), K contiguous */
    const float* bias;    /* fp32 [Cout] (folded BatchNorm shift / conv bias) or NULL */
    int32_t Cout;         /* multiple of block_n */
    int32_t block_n;      /* 32, 64, 128 or 256 */
    int32_t phases;       /* 1, or 4 for the fused nearest-x2 upsample (phase p = 2*a+b adds (a,b) to every (dh,dw)) */

    int32_t Wt, Ht, Nt;   /* tile-space extents (the pixels that produce outputs) */
    int32_t TW, TH, TN;   /* tile box, TW*TH*TN == 128 */

    /* output: pixel (n, h, w) of tile space, phase (a, b) -> out + n*pitch_n + (h*sy+a)*pitch_h + (w*sx+b)*pitch_w + c */
    void* out;            /* fp16 (mode 0) */
    int64_t out_pitch_w, out_pitch_h, out_pitch_n;
    int32_t out_sy, out_sx;
    const void* residual; /* fp16, same addressing as out, added before ReLU; or NULL */
    int32_t relu;

    /* mode 1 ("head"): block_n == Cout == 32; ReLU(acc) is contracted in fp32 with head_w [classes][32] + head_b
     * and written as fp32 NCHW logits [N][classes][Ht][Wt] to head_out (final 1x1 conv, unet.py:141) */
    int32_t mode;
    int32_t head_classes; /* <= 8 */
    const float* head_w;
    const float* head_b;
    float* head_out;

    /* 1: compute each pair of neighbouring tiles with a CTA pair (cluster of 2, tcgen05 cta_group::2; mode 0,
     * block_n >= 128): each CTA stages half of the weight tile. Same results; 0 = one CTA per tile. */
    int32_t cta_pair;

    /* Split ("strict") precision: every activation and weight is the unevaluated sum of two fp16 numbers, hi = half(v) and
     * lo = half(v - hi) (22+ significant bits), stored as two planes; the kernel accumulates hi*hi + hi*lo + lo*hi in fp32
     * (3 tensor-core MMAs per K step; the lo*lo term is below fp32 resolution). This is what meets the reference's fp32
     * results (logits 1e-3 rel, argmax identical up to the fp32 noise floor); split == 0 is the fast single-fp16 mode.
     *   srcs[i].plane        element stride between the planes of source i
     *   weights              fp16 [2][phases*Cout][K] (hi plane, then lo plane)
     *   out_plane/res_plane  element stride between the planes of out / residual
     * acc_scale (0 = 1): the fp32 accumulator is multiplied by it before bias/residual; the host pre-scales the weights by
     * its inverse (a power of two) so that the lo parts of small weights stay in fp16's normal range. */
    int32_t split;
    int64_t out_plane;
    int64_t res_plane;
    float acc_scale;

    /* K chunking (mode 0; meant for split precision with long K loops): the tensor core truncates its fp32 accumulator after
     * every MMA, so a tile's K loop is cut into chunks of `kchunk` 64-element K blocks whose results the epilogue adds with
     * round-to-nearest fp32 adds through `scratch` (>= grid x 128 x block_n x 4 bytes, see rsb_conv_scratch_bytes; private to
     * the launch, reusable by the next launch on the same stream). 0: no chunking. */
    int32_t kchunk;
    float* scratch;
    int64_t scratch_bytes;

    /* BatchNorm batch statistics fused into the epilogue (training forward of a conv that feeds nn.BatchNorm2d: torchvision
     * resnet.py Bottleneck.forward bn1-3, robosat/unet.py:122-130 in train mode). mode 0, split 0, no residual, phases 1.
     * For every tile t (flat index ((n-tile * tiles_h) + h-tile) * tiles_w + w-tile) and every 32-row quarter q of it:
     *   stats[(t*4 + q)*2*Cout + c]        = sum   of the fp16 outputs of channel c over the quarter's in-range pixels
     *   stats[(t*4 + q)*2*Cout + Cout + c] = sum of their squares
     * every entry is written exactly once per run (no zeroing needed); rsb_bn_partials_finalize folds them. NULL: off. */
    float* stats;
    int64_t stats_bytes;
} rsb_conv_desc;

typedef struct rsb_conv_plan rsb_conv_plan;

/* upper bound of the scratch a chunked plan with this block_n needs on the current device (SMs x 128 x block_n x 4 bytes) */
int64_t rsb_conv_scratch_bytes(int32_t block_n);
int rsb_conv_plan_create(const rsb_conv_desc* desc, rsb_conv_plan** out_plan);
void rsb_conv_plan_destroy(rsb_conv_plan* plan);
/* number of CTAs / tiles the plan launches (for tests and occupancy accounting) */
int rsb_conv_plan_info(const rsb_conv_plan* plan, int32_t* grid, int32_t* tiles, int32_t* kblocks, int32_t* smem_bytes);
int rsb_conv_run(const rsb_conv_plan* plan, void* stream);
/* same contraction with a plain SIMT kernel reading global memory directly (no TMA / tcgen05).
 * Test-only checker used to bisect the tensor-core path on the device; never on the product path. */
int rsb_conv_run_simt_check(const rsb_conv_desc* desc, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Line-buffer variant of the same convolution for stride-1 layers with few output channels at high resolution
 * (dec5 + final, dec4, layer1 3x3; unet.py:127, 138-141): a tile is 128 pixels of one output row, input rows live in a
 * shared-memory ring and are fetched once for all filter taps. Same arithmetic and packed weight layout
 * ([phase*Cout + co][(tap_h, tap_w)][ci]) as rsb_conv_*; see csrc/rsb_conv_row.cu.
 */
typedef struct rsb_rowconv_desc {
    rsb_conv_src src;        /* dense NHWC view of the input (TMA zero-fills outside = padding) */
    int32_t cin;             /* 32, 64 or 128 */
    int32_t taps_h, taps_w;  /* 3x3, or 2x2 for the fused upsample */
    int32_t dh0, dw0;        /* displacement of tap (0,0) for phase (0,0): -1, -1 */
    int32_t nsub;            /* 1, or 2 column phases b (phase b adds b to dw) computed per tile */
    int32_t nphase_a;        /* 1, or 2 row phases a (phase a adds a to dh), one per work unit */
    const void* weights;     /* fp16 [(a*nsub + b)*Cout + co][taps_h*taps_w*cin] */
    const float* bias;       /* fp32 [Cout] or NULL */
    int32_t Cout;            /* 32 or 64 */
    int32_t Wt, Ht, Nt;      /* tile-space extents */
    void* out;               /* fp16, addressed like rsb_conv_desc.out (mode 0) */
    int64_t out_pitch_w, out_pitch_h, out_pitch_n;
    int32_t out_sy, out_sx;
    int32_t relu;
    int32_t mode;            /* 0: fp16 NHWC output; 1: head (Cout 32 -> fp32 NCHW logits through head_w / head_b) */
    int32_t head_classes;
    const float* head_w;
    const float* head_b;
    float* head_out;
    int32_t rows_per_unit;   /* output rows per work unit (0 = default 32) */
    /* strict precision (see rsb_conv_desc.split): mode 1, cin 32, 3x3 only -- src.plane gives the lo plane of the input,
     * weights are fp16 [2][Cout][K] (hi, lo of w * 2^e), acc_scale = 2^-e */
    int32_t split;
    float acc_scale;
} rsb_rowconv_desc;

typedef struct rsb_rowconv_plan rsb_rowconv_plan;
int rsb_rowconv_plan_create(const rsb_rowconv_desc* desc, rsb_rowconv_plan** out_plan);
void rsb_rowconv_plan_destroy(rsb_rowconv_plan* plan);
int rsb_rowconv_run(const rsb_rowconv_plan* plan, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Input pre-pass. Replaces `images.to(device)` + the stem's NCHW read (predict.py:83, train.py:172) and,
 * for uint8 input, ToTensor + Normalize (predict.py:71-73). Writes the space-to-depth view the stem
 * convolution consumes: fp16 [N][H/2][W/2 + 4][16], pixel (hh, ww) at column ww + 2, channel
 * (ph*2 + pw)*3 + c = x[n, c, 2*hh+ph, 2*ww+pw]; channels 12..15 and the pad columns are zero.
 *   src_kind 0: fp32 NCHW, already normalised (the reference API)     src_kind 1: uint8 NHWC raw RGB
 */
int rsb_prepass_s2d(const void* src, int32_t src_kind, void* dst, int32_t N, int32_t H, int32_t W,
                    const float* mean3_host, const float* std3_host, void* stream);

/* strict precision: also writes the lo plane at dst + plane (elements): lo = half(x - float(half(x))) */
int rsb_prepass_s2d_split(const void* src, int32_t src_kind, void* dst, int64_t plane, int32_t N, int32_t H, int32_t W,
                          const float* mean3_host, const float* std3_host, void* stream);

/* NHWC fp16 max pooling. Replaces resnet.maxpool (unet.py:125: k3 s2 p1) and F.max_pool2d(enc4, 2, 2) (unet.py:132).
 * Output pixel pitches are explicit so the result can land inside a padded buffer. */
int rsb_maxpool_nhwc(const void* src, void* dst, int32_t N, int32_t H, int32_t W, int32_t C, int32_t k, int32_t s,
                     int32_t p, void* stream);

/* strict precision: the maximum of the (hi, lo) pairs, i.e. of the exact fp32 sums hi + lo, written as a pair again */
int rsb_maxpool_nhwc_split(const void* src, int64_t src_plane, void* dst, int64_t dst_plane, int32_t N, int32_t H, int32_t W,
                           int32_t C, int32_t k, int32_t s, int32_t p, void* stream);

/* Training-side augmentation (robosat/transforms.py:127-221 as composed in train.py:253-258): per sample an optional left-right flip
 * followed by k counter-clockwise quarter turns, applied to the RGB tile uint8 [N][S][S][3] and its mask uint8 [N][S][S] (mask may be
 * NULL); ops int32 [N] on the device, op = flip | (k << 1). out_mask is int64 (what the losses consume). Not in place. */
int rsb_augment_dihedral(const uint8_t* img, const uint8_t* mask, const int32_t* ops, uint8_t* out_img, int64_t* out_mask, int32_t N, int32_t S,
                         void* stream);

/* Predict head. Replaces softmax(outputs, 1) ... np.digitize(foreground, linspace(0,1,256)).astype(uint8)
 * (predict.py:87, 93, 98-103) for the 2-class case, including the crop of the `overlap` border (datasets.py:133-136).
 * logits fp32 [N][2][H][W] -> quant uint8 [N][H-2o][W-2o]; probs_fg (fp32, same cropped shape) optional. */
int rsb_head_quantize(const float* logits, uint8_t* quant, float* probs_fg, int32_t N, int32_t H, int32_t W,
                      int32_t overlap, void* stream);
/* softmax over C for any class count: logits fp32 [N][C][H][W] -> probs fp32 same shape (predict.py:87) */
int rsb_softmax_nchw(const float* logits, float* probs, int32_t N, int32_t C, int32_t HW, void* stream);
/* `buffer_tile_image` (robosat/tiles.py:162-227) on the device: builds B buffered tiles uint8 [B][S+2o][S+2o][3] from a cache of
 * decoded RGB tiles uint8 [slots][S][S][3]. slots: int32 [B][9] (device), row-major over (dy, dx) in {-1,0,1}^2, entry 4 = the
 * centre tile, -1 = no such neighbour (nodata 0, as the reference's Image.new(color=0)). */
int rsb_stitch_halo(const uint8_t* cache, const int32_t* slots, uint8_t* out, int32_t B, int32_t S, int32_t overlap, void* stream);
/* `rs masks` soft vote (robosat/tools/masks.py:42-84): quant uint8 [K][n] probability bins of K models (as written by rs predict),
 * weights float64 [K] on the device or NULL -> mask uint8 [n] = argmax([1 - p, p]) of the weighted average, float64, numpy's order. */
int rsb_softvote(const uint8_t* quant, const double* weights, uint8_t* mask, int32_t K, int64_t n, void* stream);
/* `rs weights` histogram (robosat/tools/weights.py:39-49): counts[c] += #(labels == c) for c < C; counts is uint64 [C] on the device */
int rsb_class_histogram(const uint8_t* labels, int64_t n, int32_t C, uint64_t* counts, void* stream);
/* `Predictor.segment` head (robosat/tools/serve.py:150-165): output.argmax(axis=0).astype(uint8) of fp32 NCHW logits
 * -> uint8 [N][H*W] class indices, first maximum wins like np.argmax; C <= 255. */
int rsb_head_argmax(const float* logits, uint8_t* mask, int32_t N, int32_t C, int32_t HW, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Host-side PNG codec for the files either side of the predict path (HOST pointers, plain C over zlib, no Python / GIL so the
 * tools' pool threads run truly in parallel). Pixel-identical to PIL; not a compute fallback -- no device work happens here.
 */
/* `Image.open(path).convert("RGB")` (robosat/tiles.py:150-159,181) for 8-bit non-interlaced PNGs (gray, RGB, palette, +alpha):
 * out_rgb_host uint8 [h][w][3]. RSB_E_UNSUPPORTED for other PNG flavours / non-PNG files (the caller then uses PIL). */
/* zlib-wrapped DEFLATE stream (RFC 1950 / 1951; what PNG IDAT chunks carry) -> exactly out_len bytes, Adler-32 verified, with the
 * library's own decoder (csrc/rsb_inflate.cpp); RSB_E_INVALID for anything it rejects (the PNG reader then asks zlib). */
int rsb_zlib_inflate(const uint8_t* stream_host, int64_t n, uint8_t* out_host, int64_t out_len);
int rsb_png_decode_rgb(const uint8_t* file_bytes_host, int64_t n, uint8_t* out_rgb_host, int32_t w_expected, int32_t h_expected);
int rsb_png_read_rgb(const char* path, uint8_t* out_rgb_host, int32_t w_expected, int32_t h_expected);
/* `Image.fromarray(q, mode="P"); putpalette(palette); save(path)` (robosat/tools/predict.py:105-113): 8-bit palette PNG,
 * palette_rgb_host uint8 [entries][3]; level = zlib level (0-9, <0 default). Noise-like rasters (a level-1 probe of 16 rows does not
 * shrink below 90 %) are coded with zlib's Z_RLE strategy: same size, a third of the time. encode returns the byte count or a
 * negative code. */
int64_t rsb_png_encode_p8(const uint8_t* pixels_host, int32_t w, int32_t h, const uint8_t* palette_rgb_host, int32_t entries, int32_t level,
                          uint8_t* out_host, int64_t capacity);
int rsb_png_write_p8(const char* path, const uint8_t* pixels_host, int32_t w, int32_t h, const uint8_t* palette_rgb_host, int32_t entries,
                     int32_t level);

/* Whole-batch variants, fanned out over `threads` threads inside the library (one call per tile batch from the tools):
 * read: rcs_host[i] receives the per-file code (RSB_E_UNSUPPORTED entries are left for another decoder); the return value is the
 * worst real error. write: image i is pixels_host + i*image_stride; make_dirs != 0 creates the parent directories (z/x/). */
int rsb_png_read_rgb_batch(const char* const* paths, int32_t n, uint8_t* const* outs_rgb_host, int32_t w_expected, int32_t h_expected,
                           int32_t threads, int32_t* rcs_host);
int rsb_png_write_p8_batch(const char* const* paths, int32_t n, const uint8_t* pixels_host, int64_t image_stride, int32_t w, int32_t h,
                           const uint8_t* palette_rgb_host, int32_t entries, int32_t level, int32_t threads, int32_t make_dirs);

/* ---------------------------------------------------------------------------------------------
 * Losses and metrics on fp32 NCHW logits + int64 targets [N][H][W].
 */
/* CrossEntropyLoss2d.forward (losses.py:24-25): weighted NLL of log_softmax, mean over sum of target weights.
 * loss_out: fp32 scalar; grad (optional, fp32 NCHW) receives dLoss/dlogits. weight may be NULL (all ones).
 * scratch: >= 2 doubles, zeroed by the call. */
int rsb_cross_entropy(const float* logits, const int64_t* targets, const float* weight, float* loss_out, float* grad,
                      double* scratch, int32_t N, int32_t C, int32_t HW, void* stream);

/* FocalLoss2d.forward (losses.py:49-50): NLLLoss(weight)((1 - softmax)^gamma * log_softmax, targets) + gradient. scratch: 2 doubles. */
int rsb_focal(const float* logits, const int64_t* targets, const float* weight, float gamma, float* loss_out, float* grad,
              double* scratch, int32_t N, int32_t C, int32_t HW, void* stream);
/* mIoULoss2d.forward (losses.py:71-83): max(1 - mean_{c,n} soft-IoU, weighted cross entropy); the gradient is the one of
 * whichever term is larger (decided on the device, no host synchronisation). scratch: rsb_miou_scratch_doubles(N, C) doubles. */
int64_t rsb_miou_scratch_doubles(int32_t N, int32_t C);
int rsb_miou(const float* logits, const int64_t* targets, const float* weight, float* loss_out, float* grad, double* scratch,
             int32_t N, int32_t C, int32_t HW, void* stream);

/* LovaszLoss2d.forward (losses.py:96-119) and its closed-form gradient (SURVEY.md A8), per image:
 * errors e = 1 - (2*onehot-1)*x over the flattened C*H*W vector, descending sort, Jaccard gradient, dot(relu(e), J).
 * workspace: rsb_lovasz_workspace_bytes(N, C, HW) bytes. loss_out: fp32 scalar (mean over N). grad optional. */
int64_t rsb_lovasz_workspace_bytes(int32_t N, int32_t C, int32_t HW);
int rsb_lovasz(const float* logits, const int64_t* targets, float* loss_out, float* grad, void* workspace,
               int64_t workspace_bytes, int32_t N, int32_t C, int32_t HW, void* stream);

/* Metrics.add (metrics.py:27-41) for a whole batch: counts[4] += {tn, fn, fp, tp} with the reference's
 * argmax / (pred/actual in {NaN, inf, 0, 1}) semantics. counts: int64[4] on the device, accumulated. */
int rsb_metrics_count(const float* logits, const int64_t* targets, int64_t* counts, int32_t N, int32_t C, int32_t HW,
                      void* stream);

/* torch.optim.Adam.step (train.py:81,188) over one flat fp32 parameter arena:
 * betas (b1,b2), eps, no weight decay, no amsgrad; `step` is the 1-based step count for bias correction. */
int rsb_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float b1,
                  float b2, float eps, int32_t step, void* stream);

/* Same update behind an overflow guard for mixed-precision training (no host synchronisation): if `grad` holds an inf / NaN the
 * whole step is skipped on the device (parameters and moments untouched). guard_state: int32[4] on the device, zero-initialised by
 * the caller once -- [0] scratch flag, [1] steps skipped so far (bias corrections use step - skipped), [2] flag of the last
 * finished step (poll it to adapt the loss scale), [3] steps seen. With no skipped step the result equals rsb_adam_step bit for bit. */
int rsb_adam_step_guarded(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float b1,
                          float b2, float eps, int32_t step, int32_t* guard_state, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Training path (robosat/tools/train.py:163-201: net.train() forward, loss.backward()). Activations and activation
 * gradients are NHWC fp16 [M = N*H*W][C]; gradients carry the caller's loss scale; parameter gradients are fp32, unscaled.
 */
/* train-mode BatchNorm2d (torchvision resnet50 inside unet.py:122-130): batch sums -> statistics / running-stat update -> apply.
 * sums: 20*C doubles of scratch (8 replicated accumulator slots, arrival counter, backward coefficients). finalize writes mean, invstd, scale = gamma*invstd, shift = beta - mean*scale and updates
 * running_mean / running_var (unbiased, momentum) / num_batches_tracked when those pointers are non-NULL. */
int rsb_bn_stats(const void* z, double* sums, int64_t M, int32_t C, void* stream);
int rsb_bn_finalize(const double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                    int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int32_t C, int64_t M, float eps,
                    float momentum, void* stream);
/* rsb_bn_stats + rsb_bn_finalize in one launch (the last block of the reduction does the per-channel epilogue) */
int rsb_bn_stats_finalize(const void* z, double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                          int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int64_t M, int32_t C, float eps,
                          float momentum, void* stream);
/* "_chained" variants (what the training plan uses): the same arithmetic, but (a) launched with programmatic stream serialization
 * so a chain of small kernels does not pay a full launch gap per link, and (b) without the per-call memset: `sums` must be
 * zero-initialised ONCE by the caller and is left zeroed by the reduction's last block. */
int rsb_bn_stats_finalize_chained(const void* z, double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                                  int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int64_t M, int32_t C, float eps,
                                  float momentum, void* stream);
/* Same statistics / finalize from the per-quarter-tile partial sums a convolution wrote through rsb_conv_desc.stats
 * (partials: fp32 [rows][2][C], rows = spatial tiles * 4) instead of re-reading z: 1/8 of the bytes. `chained` as above
 * (1: no memset, programmatic stream serialization; sums must be zero on entry and is left zeroed). */
int rsb_bn_partials_finalize(const float* partials, int64_t rows, double* sums, const float* gamma, const float* beta, float* running_mean,
                             float* running_var, int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int64_t M,
                             int32_t C, float eps, float momentum, int32_t chained, void* stream);
int rsb_bn_apply_chained(const void* z, const float* scale, const float* shift, const void* residual, void* y, int64_t M, int32_t C,
                         int32_t relu, void* stream);
int rsb_bn_backward_chained(const void* dy, const void* y, const void* z, const float* mean, const float* invstd, const float* gamma,
                            const float* mask_scale, const float* mask_shift, double* sums, void* dz, void* g_out, float* dgamma, float* dbeta,
                            float inv_loss_scale, int64_t M, int32_t C, void* stream);
/* y = relu?(z*scale + shift (+ residual)) */
int rsb_bn_apply(const void* z, const float* scale, const float* shift, const void* residual, void* y, int64_t M, int32_t C,
                 int32_t relu, void* stream);
/* autograd of relu(bn(z) (+ identity)): g = dy * (y > 0) (y NULL: no mask); dz = gamma*invstd*(g - mean(g) - zhat*mean(g*zhat));
 * g_out (optional) receives g = the gradient of the identity branch; dgamma/dbeta fp32 multiplied by inv_loss_scale.
 * mask_scale / mask_shift (with y NULL): the output was the plain y = half(relu(z*scale + shift)) of rsb_bn_apply, so its ReLU mask
 * is re-derived from z (bit-identical: half(o) > 0 <=> o > 2^-25) and y is not read at all. */
int rsb_bn_backward(const void* dy, const void* y, const void* z, const float* mean, const float* invstd, const float* gamma,
                    const float* mask_scale, const float* mask_shift, double* sums, void* dz, void* g_out, float* dgamma, float* dbeta,
                    float inv_loss_scale, int64_t M, int32_t C, void* stream);
/* out = (a (+ b)) * (y > 0): ReLU backward with optional gradient fan-in (skip connections); y NULL: plain sum */
int rsb_relu_backward(const void* a, const void* b, const void* y, void* out, int64_t n, void* stream);
/* autograd of max_pool2d (unet.py:125, :132) on NHWC fp16: first maximum of every window receives its gradient.
 * argmax_scratch: N*OH*OW*C bytes of device scratch (one window position per pooled element) -> two streaming passes;
 * NULL -> single-pass kernel that re-derives the argmax per input pixel (slower, no scratch). Same results. */
int rsb_maxpool_backward(const void* x, const void* dy, void* dx, void* argmax_scratch, int32_t N, int32_t H, int32_t W, int32_t C,
                         int32_t k, int32_t s, int32_t p, void* stream);
/* autograd's AccumulateGrad for every parameter at once (loss.backward(), train.py:186): dst_i[0:n_i] += alpha * src_i[0:n_i]
 * for `segments` rows (src pointer, dst pointer, n_i <= 2^31) of a device-resident int64 table; fp32, one block per row. */
int rsb_multi_axpy(const int64_t* table, int32_t segments, float alpha, void* stream);
/* final 1x1 conv 32 -> classes with bias (unet.py:141) as its own step in training: fp32 NCHW logits from NHWC fp16 dec5 */
int rsb_final_forward(const void* y5, const float* w, const float* b, float* logits, int32_t N, int32_t HW, int32_t classes,
                      void* stream);
/* its autograd: dy5 (fp16, times loss_scale), dW [classes][32], db [classes] (fp32, unscaled). acc: classes*32 + 8 doubles. */
int rsb_final_backward(const float* dlogits, const void* y5, const float* w, void* dy5, double* acc, float* dw, float* db,
                       float loss_scale, int32_t N, int32_t HW, int32_t classes, void* stream);
/* fp32 OIHW master weights -> fp16 packed operand matrix: dst[i] = half(sum of src[map4[4i..4i+3]] (entries < 0 skipped)) */
int rsb_pack_weights(const float* src, const int32_t* map4, void* dst, int64_t n, void* stream);
/* the same with ONE source index per packed element (map1: int32 [n], -1 = zero; n a multiple of 8, map1 and dst 16-byte
 * aligned): a quarter of the map bytes; used for every layout but the pre-summed nearest-x2 taps */
int rsb_pack_weights1(const float* src, const int32_t* map1, void* dst, int64_t n, void* stream);
/* packed fp32 gradient -> OIHW fp32 gradient: grad[map4[4i+j]] += packed_grad[i] * mul (the transpose of rsb_pack_weights) */
int rsb_unpack_grads(const float* packed_grad, const int32_t* map4, float* grad, int64_t n, float mul, void* stream);

/* the same reduction without atomics (deterministic): element i of the compact list writes grad[dst_idx[i]] = mul * (sum of the
 * packed gradient elements inv4[4i..4i+3], entries < 0 skipped, added in index order); inv4 is the inverse of map4 */
int rsb_unpack_grads_gather(const float* packed_grad, const int32_t* dst_idx, const int32_t* inv4, float* grad, int64_t n, float mul,
                            void* stream);

/* Strict-precision training forward (the opt-in `strict` training plan): forward activations are fp16 (hi, lo) pairs in two
 * planes `plane` elements apart (value = hi + lo, exact in fp32; hi = half(v), lo = half(v - hi)), as the split convolutions
 * (rsb_conv_desc.split) read and write them. The backward keeps single fp16 operands and reads the hi planes.
 *
 * fp32 OIHW master weights -> split packed operand: dst[i] = hi, dst[plane + i] = lo of (sum of the map's sources) * scale, scale a
 * power of two fixed per layer (the conv's acc_scale is its inverse). Every element whose scaled hi is not a finite fp16 adds one to
 * *overflow (int32 on the device, never reset by the call): the weights have outgrown the layer's exponent. map4 / map1 as in
 * rsb_pack_weights / rsb_pack_weights1 (the 1-index form: n and plane multiples of 8, map and dst 16-byte aligned). */
int rsb_pack_weights_split(const float* src, const int32_t* map4, void* dst, int64_t plane, int64_t n, float scale, int32_t* overflow,
                           void* stream);
int rsb_pack_weights1_split(const float* src, const int32_t* map1, void* dst, int64_t plane, int64_t n, float scale, int32_t* overflow,
                            void* stream);
/* rsb_bn_stats_finalize on a two-plane z: the batch sums of hi + lo and of its square are accumulated in fp64 from the first add.
 * Same sums scratch, outputs and running-stat update; "_chained" as rsb_bn_stats_finalize_chained (sums zero on entry, left zeroed).
 * overflow (optional): the pack's counter; while it is non-zero the running statistics and num_batches are left untouched. */
int rsb_bn_stats_finalize_split(const void* z, int64_t plane, double* sums, const float* gamma, const float* beta, float* running_mean,
                                float* running_var, int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int64_t M,
                                int32_t C, float eps, float momentum, const int32_t* overflow, void* stream);
int rsb_bn_stats_finalize_split_chained(const void* z, int64_t plane, double* sums, const float* gamma, const float* beta, float* running_mean,
                                        float* running_var, int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift,
                                        int64_t M, int32_t C, float eps, float momentum, const int32_t* overflow, void* stream);
/* y = relu?(z*scale + shift (+ residual)) in fp32 from two-plane z / residual, written as a (hi, lo) pair */
int rsb_bn_apply_split(const void* z, int64_t z_plane, const float* scale, const float* shift, const void* residual, int64_t res_plane, void* y,
                       int64_t y_plane, int64_t M, int32_t C, int32_t relu, void* stream);
int rsb_bn_apply_split_chained(const void* z, int64_t z_plane, const float* scale, const float* shift, const void* residual, int64_t res_plane,
                               void* y, int64_t y_plane, int64_t M, int32_t C, int32_t relu, void* stream);
/* rsb_maxpool_backward for a two-plane x: every window's gradient goes to the FIRST position (row-major scan) whose hi + lo equals
 * the window maximum, the element rsb_maxpool_nhwc_split forwarded (ATen's tie rule on the fp32 values). dy / dx single fp16;
 * argmax_scratch (N*OH*OW*C bytes) is required. */
int rsb_maxpool_backward_split(const void* x, int64_t x_plane, const void* dy, void* dx, void* argmax_scratch, int32_t N, int32_t H, int32_t W,
                               int32_t C, int32_t k, int32_t s, int32_t p, void* stream);
/* rsb_final_forward on two-plane dec5 activations: hi + lo contracted with the fp32 weights in fp32. overflow (optional): the pack's
 * counter; while it is non-zero every logit is NaN, so that the step's loss and gradients are not finite (a guarded optimiser skips it) */
int rsb_final_forward_split(const void* y5, int64_t plane, const float* w, const float* b, const int32_t* overflow, float* logits, int32_t N,
                            int32_t HW, int32_t classes, void* stream);

/* Weight gradient of the convolution described by `fwd` (same sources / segments / phases / tile space), on tensor cores:
 *   dw_packed[phase*Cout + co][k] = sum_pixels dy_phase[pixel][co] * x_segment(k)[pixel + (dh,dw)][k % 64-block]   (fp32)
 * i.e. the gradient in the forward kernel's packed weight layout (rsb_unpack_grads folds it back to OIHW).
 * dy is addressed like fwd->out (same pitches / phase strides). Replaces autograd's conv weight gradients (train.py:186). */
typedef struct rsb_wgrad_plan rsb_wgrad_plan;
int rsb_wgrad_plan_create(const rsb_conv_desc* fwd, const void* dy, float* dw_packed, rsb_wgrad_plan** out_plan);
/* Deterministic split-K: bytes of scratch the plan needs (0 when it has a single pixel slice), and the call that hands it over.
 * With a scratch every slice stores its partial gradient and a second kernel adds the slices in index order (bit-identical from
 * run to run); without one the slices add into dw_packed with fp32 atomics. The scratch is private to a launch and may be shared
 * by all plans that run on one stream. */
int64_t rsb_wgrad_plan_scratch_bytes(const rsb_wgrad_plan* plan);
int rsb_wgrad_plan_set_scratch(rsb_wgrad_plan* plan, float* scratch, int64_t scratch_bytes);
void rsb_wgrad_plan_destroy(rsb_wgrad_plan* plan);
int rsb_wgrad_run(const rsb_wgrad_plan* plan, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RSB200_H */
