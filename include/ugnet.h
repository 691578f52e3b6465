/* ugnet.h — C ABI of libugnet.so: the B200 (sm_100a) engine for the two-stage hot path of
 * BY-Elysia/UNet-GooLeNet (UNet forward -> mask -> bbox -> ROI crop/resize -> GoogLeNet forward).
 *
 * The reference is pure Python and has no FFI of its own; its "interface" for this path is
 *   nets.basicUnet.UNetTaskAligWeight.forward          (分割/nets/basicUnet.py:406-437)
 *   nets.tasks.TransformerDecoder.forward              (分割/nets/tasks.py:218-231)
 *   util.roi.process_and_augment_roi                   (分类/util/roi.py:12-51)
 *   GoogLeNetClassifier.forward / torchvision GoogLeNet (分类/test.py:64-73)
 *   inference_all                                      (分类/test.py:74-96, 分割/predict.py:11-51)
 * The Python shells in unet-goolenet_b200/ keep those names and lower each forward into a list of the ops
 * declared here (a "program"), which the engine executes on one CUDA stream.  Grad-CAM of the classifier at inception5b
 * (pytorch-grad-cam's GradCAM on model.googlenet.inception5b) is one more op, ug_cam, which programs built with
 * cam=True append after the head; ug_source_frame, which programs built with source_frame=True append last, carries the
 * mask, the box and the map to each source image's own size.  Every entry point:
 *   - takes raw device pointers and explicit shapes, never owns caller memory, never throws;
 *   - returns UG_OK (0) or a negative UG_E* code; the message is available via ug_last_error();
 *   - is asynchronous on the given stream (cudaStream_t passed as void*), except *_host helpers;
 *   - is not thread-safe per handle (one handle per device/thread).
 * All activations are NHWC bf16 unless stated; all folded scale/bias vectors are fp32.
 */
#ifndef UGNET_H_
#define UGNET_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UG_VERSION 100

enum { UG_OK = 0, UG_EINVAL = -1, UG_ECUDA = -2, UG_ENOMEM = -3, UG_EUNSUPPORTED = -4 };
enum { UG_ACT_NONE = 0, UG_ACT_RELU = 1, UG_ACT_GELU = 2 };
enum { UG_EPI_STORE = 0, UG_EPI_ADD = 1, UG_EPI_GATE = 2, UG_EPI_OUTC = 3 };

typedef struct ug_engine* ug_handle;
typedef struct ug_program_s* ug_program;

/* ---- implicit-GEMM convolution / linear layer on tcgen05 tensor cores --------------------------------
 * Replaces nn.Conv2d(3x3,p=1)+BatchNorm2d+ReLU (basicUnet.py:25-40), Conv2dReLU (tasks.py:98-120),
 * nn.ConvTranspose2d(2,2,s=2) (basicUnet.py:121), nn.Linear (tasks.py:50-53,66-72,127-131),
 * outc 1x1 (basicUnet.py:391,435) and torchvision BasicConv2d.  Stride is always 1 and 2*pad == R-1.
 * in : pixel (n,y,x) at in + ((n*H+y)*W+x)*in_cstride, channels [0,Cin)   (channel-slice views allowed)
 * w  : bf16 [Npad][R*S*Cin_pad], K index = (r*S+s)*Cin_pad + c, Cin_pad = round_up(Cin,64), zero padded
 * out: value(n,y,x,j) = act(acc*scale[j] + bias[j]) then the epilogue `mode`:
 *   UG_EPI_STORE: out[((n*OH+oy)*OW+ox)*out_cstride + c] (bf16)
 *   UG_EPI_ADD  : ... + add[n*add_bstride + (oy*OW+ox)*add_cstride + c]           (residual / pos-embedding)
 *   UG_EPI_GATE : add[...] + value*(1+gate[n*N+c])        (CoordAtt3: e_1 + g*def_d + def_d, basicUnet.py:229)
 *   UG_EPI_OUTC : logits[(n*H+y)*W+x] = sum_j value_j*outc_w[j] + outc_b; mask = sigmoid(logit) > 0.5
 *                 (outc + roi.py:22-23); nothing is written to `out`.  Requires N <= BN.
 * up == 1: (oy,ox,c) = (y,x,j).  up == 2 (ConvTranspose 2x2 s2): N = 4*convt_cout, q = j/convt_cout,
 *   (oy,ox,c) = (2y + (q>>1), 2x + (q&1), j % convt_cout).
 */
typedef struct ug_conv_desc {
  const void* in;
  int in_cstride, Cin;
  int B, H, W;
  int R, S, pad;
  const void* w;
  int N;
  const float* scale; /* may be NULL (= 1) */
  const float* bias;  /* may be NULL (= 0) */
  int act, mode;
  void* out;
  int out_cstride;
  int up, convt_cout;
  const void* add;
  long long add_bstride;
  int add_cstride;
  const float* gate;
  const float* outc_w;
  float outc_b;
  float* logits;
  unsigned char* mask;
  void* pool_out;             /* optional (3x3 multi-issuer kernel, STORE epilogue, H and W even): also write
                                 nn.MaxPool2d(2) of the output (basicUnet.py:47 DownBlock) to
                                 pool_out[((n*H/2+y)*W/2+x)*pool_cstride + c], fused into the epilogue */
  int pool_cstride;
  float* stats_sum;           /* optional (3x3 multi-issuer kernel, STORE epilogue): per-tile partial channel sums and */
  float* stats_max;           /* maxima of the stored output, [B][stats_tiles][N] fp32 — stage 1 of CoordAtt3's
                                 AdaptiveAvg/MaxPool2d(1) (basicUnet.py:217-218) fused into the epilogue; fold with
                                 ug_gate (splits = stats_tiles).  Deterministic (no atomics). */
  int stats_tiles;            /* must equal ceil(W/8) * ceil(H/16) (pixel tiles per image); checked */
  void* out2;                 /* optional second destination (1x1 layers, STORE epilogue): GEMM columns [0, n1) go to */
  int out2_cstride;           /* `out`, columns [n_split, N) to out2[... * out2_cstride + (j - n_split)]; columns */
  int n_split, n1;            /* [n1, n_split) are padding (zero weight rows), n_split % 64 == 0.  Used for the three
                                 1x1 convolutions of an Inception block that read the same tensor (torchvision
                                 Inception.forward: branch1, branch2[0], branch3[0]) as ONE GEMM: branch1 lands in the
                                 block's concat output, the two reduce results in a scratch tensor */
  long long in_rstride;       /* optional explicit input strides in elements (0 = dense: W*in_cstride, H*W*in_cstride). */
  long long in_bstride;       /* With in_cstride < Cin the 64-channel rows of neighbouring pixels OVERLAP (a TMA tensor
                                 map with a pixel stride below its inner box): together with R > 1, S == 1, pad == 0
                                 ("row taps": out(y,x) = sum_r W_r . in(y+r, x), input map H+R-1 rows, Cin <= 64) this
                                 runs a KxK strided stem convolution as a regular implicit GEMM over a space-to-depth
                                 image (GoogLeNet conv1 7x7 s2 = 4 row taps x [4 px x 16 ch] windows, see ug_s2d_desc) */
  int TW, TH, TN, BN, stages; /* tiling; 0 = engine chooses */
  int variant;                /* 0 = auto; 1 = one tile per CTA; 2 = persistent kernel (TMEM multi-buffered
                                 accumulators, TMA-store epilogue); 5 = 3x3 multi-issuer kernel (one CTA per
                                 SM, two MMA-issuing warps sharing resident or streamed weights, activation
                                 halo tile fetched once per 64-channel chunk for all nine taps; see
                                 csrc/conv_multi.cu); 6 = CTA-pair kernel (csrc/conv_pair.cu: clusters of two CTAs,
                                 tcgen05.mma.cta_group::2 with M = 256 over both SMs, each CTA holding half of the
                                 weight rows; 3x3 ReLU layers with N <= 64, STORE / OUTC / GATE epilogues);
                                 7 = the multi-issuer kernel in CTA-pair mode (3x3 ReLU layers with 128-column
                                 n-tiles, STORE / GATE epilogues; each CTA streams half of every weight tile).
                                 0 picks by the measured static rule of csrc/conv_gemm.cu (conv_prepare).
                                 Any other value is rejected with UG_EINVAL */
} ug_conv_desc;

/* Max pooling on NHWC bf16 with -inf padding (nn.MaxPool2d(2), basicUnet.py:47; torchvision GoogLeNet
 * maxpool1-4 and Inception branch4 with ceil_mode=True: caller passes the ceil-mode OH/OW).  C and both channel
 * strides are multiples of 8 and in / out are 16-byte aligned (8-channel vector accesses). */
typedef struct ug_pool_desc {
  const void* in;
  int in_cstride;
  void* out;
  int out_cstride;
  int C, B, H, W, OH, OW, k, stride, pad;
} ug_pool_desc;

/* nn.LayerNorm(C) over the last dim of [M][C] bf16 tokens (tasks.py:161-164), fp32 statistics.  C is 256, 512, 768
 * or 1024; in / out / gamma / beta are 16-byte aligned. */
typedef struct ug_layernorm_desc {
  const void* in;
  void* out;
  const float* gamma;
  const float* beta;
  int M, C;
  float eps;
} ug_layernorm_desc;

/* softmax(q k^T * scale) v per (image, head), dim_head = 64 (tasks.py:132-147 and :73-96).
 * q/k/v rows are tokens (b*S + i) with the given row strides (elements); head h uses columns [64h,64h+64).  Every row
 * stride is a multiple of 8 and at least 64*heads; k and v are 16-byte aligned, q and out 4-byte aligned. */
typedef struct ug_attn_desc {
  const void* q;
  const void* k;
  const void* v;
  int q_stride, k_stride, v_stride;
  void* out;
  int out_stride;
  int B, S, heads;
  float scale;
  int variant; /* reserved, must be 0.  S <= 208 (the 14x14 bottleneck has S = 196); longer sequences are rejected */
} ug_attn_desc;

/* AdaptiveAvgPool2d(1)/AdaptiveMaxPool2d(1) of an NHWC bf16 map (basicUnet.py:217-218), stage 1: each of
 * `splits` blocks per image reduces a contiguous pixel range to fp32 partial sums / maxima
 * psum,pmax: [B][splits][C].  Deterministic (no atomics); stage 2 lives in the gate op.  C = 8*2^k <= 512,
 * in_cstride a multiple of 8, in 16-byte aligned. */
typedef struct ug_chanstats_desc {
  const void* in;
  int in_cstride, C, B, HW, splits;
  float* psum;
  float* pmax;
} ug_chanstats_desc;

/* avg = sum(psum)/HW, max = max(pmax);  g = sigmoid(W3 (relu(W1 avg + b1) + relu(W2 max + b2)) + b3)
 * (basicUnet.py:220-225); fp32.  w1,w2: [C/2][C]; w3: [C][C/2]; g: [B][C]. */
typedef struct ug_gate_desc {
  const float* psum;
  const float* pmax;
  const float *w1, *b1, *w2, *b2, *w3, *b3;
  float* g;
  int B, C, HW, splits;
  float* hid; /* scratch fp32 [B][C/2] (hidden layer, written then read by the two launches of this op) */
} ug_gate_desc;

/* mask u8 [B,H,W] -> boxes int32 [B][4] = {x_min, y_min, x_max, y_max} with roi.py:25-36 semantics
 * (padding, clamp, end-exclusive max, centred fallback for an empty mask). */
typedef struct ug_bbox_desc {
  const unsigned char* mask;
  int* boxes;
  int B, H, W, padding;
} ug_bbox_desc;

/* roi.py:39-44 + data_utils.py:102,146-147: crop img[:, y0:y1, x0:x1] (fp32 NCHW in [0,1]) -> trunc(x*255)
 * uint8 -> channel flip (c -> 2-c) -> PIL-exact bilinear resize (horizontal pass then vertical pass,
 * 22-bit fixed point, uint8 intermediate) to SxS.  out_u8: [B][S][S][3] (HWC). */
typedef struct ug_cropresize_desc {
  const float* img;
  const int* boxes;
  unsigned char* out_u8;
  int B, H, W, S;
} ug_cropresize_desc;

/* Stem convolution fused with its im2col (no im2col matrix in HBM), N = 64 output channels, folded BN + ReLU:
 *   kind 0: UNet inc (basicUnet.py:409; ConvBatchNorm :25-40): 3x3 s1 p1 on in_f32 = fp32 NCHW [B,3,H,W]
 *           (also performs x.float(), :408); w = bf16 [64][64], column (r*3+s)*3+c, columns 27.. zero.
 * Any other kind is rejected with UG_EINVAL (GoogLeNet conv1 runs as ug_s2d_pack + a row-tap conv).
 * out: bf16 NHWC [B,H,W,out_cstride], channels [0,64). */
typedef struct ug_stem_desc {
  int kind;
  const float* in_f32;
  const unsigned char* in_u8;   /* unused */
  const void* w;
  const float* scale;
  const float* bias;
  void* out;
  int out_cstride;
  int B, H, W;
  void* pool_out;   /* optional (H and W even): also write nn.MaxPool2d(2) of the output (DownBlock,
                       basicUnet.py:47) to bf16 NHWC [B,H/2,W/2,pool_cstride], fused into the epilogue */
  int pool_cstride;
} ug_stem_desc;

/* Space-to-depth pack for GoogLeNet conv1 (torchvision BasicConv2d 7x7 s2 p3; 分类/test.py:68-73): the uint8 HWC crop
 * [B,S,S,3] (or a float NCHW image in [0,1]) -> bf16 [B][S/2+3][S/2+3][16]:
 *   q[n][Y][X][(dy*2+dx)*3 + c] = T(img[n][2Y+dy-3][2X+dx-3][c])  (0 outside the image: padding after the affine),
 *   T = to_tensor (/255) followed by torchvision's _transform_input; channels 12..15 are zero.
 * Then conv1(y,x) = sum_{r2<4} sum_{s2<4} W2[r2][s2] . q[y+r2][x+s2]: with in_cstride = 16 the 64-element window
 * q[y+r2][x .. x+3] is ONE overlapping 128-byte row of a TMA tensor map, so the layer runs on the implicit-GEMM kernel
 * with four row taps (K = 4 x 64, ug_conv_desc.in_rstride) and no thread-built im2col. */
typedef struct ug_s2d_desc {
  const unsigned char* in_u8;
  const float* in_f32;
  void* out;
  int B, S;
} ug_s2d_desc;

/* Device front-end (SURVEY §8f.1): the reference's CDDataAugmentation.transform live lines
 * (分类/util/data_utils.py:146-147, 分割/util/data_utils.py): F.resize(PIL image, (S,S), BILINEAR) + F.to_tensor.
 * src: uint8 HWC [B][Hs][Ws][3] of any size up to 8*S per side (e.g. the 512x512 sources of BASELINE config 5);
 * Pillow's antialiased resample is restated bit-exactly (support = max(in/out, 1), horizontal pass then vertical
 * pass, 22-bit fixed point, uint8 intermediate).  out_f32: fp32 NCHW [B][3][S][S] = value / 255 (the UNet input);
 * out_u8 (optional): the resized uint8 HWC image [B][S][S][3].  Either output may be NULL, not both. */
typedef struct ug_resize_desc {
  const unsigned char* src;
  float* out_f32;
  unsigned char* out_u8;
  int B, Hs, Ws, S;
} ug_resize_desc;

/* `wavelet_enhance` (分类/test.py:17-63; SURVEY §8f.2): grayscale uint8 [B][H][W] -> pseudo-RGB uint8 HWC [B][H][W][3]:
 * R = normalize(image), G = normalize(resize(cA)), B = normalize(resize(sqrt(cH^2+cV^2+cD^2))) with the single-level
 * Haar transform of PyWavelets (float32, 'symmetric' extension), cv2.resize INTER_LINEAR back to HxW and
 * normalize(x) = ((x - min) / max(x - min) * 255).astype(uint8) per image.  workspace: device scratch of at least
 * ug_wavelet_workspace_bytes(B, H, W) bytes.  Five small launches on the stream. */
typedef struct ug_wavelet_desc {
  const unsigned char* gray;
  unsigned char* out_u8;
  void* workspace;
  size_t workspace_bytes;
  int B, H, W;
} ug_wavelet_desc;

/* Ragged batches: B images of different sizes packed back to back in one uint8 buffer, described by a device table of
 * B entries (16 bytes each).  Image i's grayscale bytes start at byte px_offset of the packed buffer, its HWC RGB bytes
 * at byte 3 * px_offset, so one table describes the gray input of ug_wavelet_ragged, its RGB output and the RGB input
 * of ug_resize_ragged.  The table is input from outside the library (a plan image's host fills it): every kernel
 * checks each entry before touching memory.  An entry with a negative offset, a side out of range or an extent past the
 * buffer's capacity is "bad": the kernel reads nothing for it and sets status[i] = 1 (status[i] = 0 otherwise; status
 * is an optional int32 [B]).  Packing, validation and chunking live in unet-goolenet_b200/util/ragged.py. */
typedef struct ug_ragged_image {
  long long px_offset;
  int H, W;
} ug_ragged_image;

/* ug_resize_desc over a ragged batch of uint8 HWC sources: image i is index[i].H x index[i].W at src + 3*px_offset,
 * 1 <= H, W <= 8*S, and 3*(px_offset + H*W) <= src_bytes.  Same arithmetic and outputs as ug_resize_desc (one launch,
 * launch geometry sized for the largest source the descriptor allows, so it does not depend on the table).  A bad entry
 * writes zeros to image i's outputs. */
typedef struct ug_resize_ragged_desc {
  const unsigned char* src;
  const ug_ragged_image* index; /* device, [B] */
  int* status;                  /* optional int32 [B] */
  float* out_f32;
  unsigned char* out_u8;
  long long src_bytes;
  int B, S;
} ug_resize_ragged_desc;

/* ug_wavelet_desc over a ragged batch of grayscale images: image i is index[i].H x index[i].W (H, W in [2, 32768]) at
 * gray + px_offset with px_offset + H*W <= capacity_px; its pseudo-RGB result goes to out_u8 + 3*px_offset (out_u8
 * holds 3*capacity_px bytes).  workspace: at least ug_wavelet_ragged_workspace_bytes(B, capacity_px) bytes.  A bad entry
 * has no trustworthy destination: nothing is written for it except its status. */
typedef struct ug_wavelet_ragged_desc {
  const unsigned char* gray;
  const ug_ragged_image* index; /* device, [B] */
  int* status;                  /* optional int32 [B] */
  unsigned char* out_u8;
  void* workspace;
  size_t workspace_bytes;
  long long capacity_px;
  int B;
} ug_wavelet_ragged_desc;

/* AdaptiveAvgPool2d(1) + Linear(C, ncls): in NHWC bf16 [B][HW][C], w fp32 [ncls][C], logits fp32 [B][ncls].  C is
 * even and at most 1024, in is 4-byte aligned (read as bf16 pairs). */
typedef struct ug_head_desc {
  const void* in;
  const float* w;
  const float* b;
  float* logits;
  int B, HW, C, ncls;
} ug_head_desc;

/* Grad-CAM at GoogLeNet's inception5b (pytorch-grad-cam's GradCAM(model, target_layers=[model.googlenet.inception5b])).
 * torchvision's GoogLeNet ends in avgpool(h x w) -> flatten -> dropout (identity in eval) -> fc, so the gradient of
 * logit c with respect to feat[y][x][k] is W[c][k] / (h*w) at every position: the Grad-CAM channel weights need no
 * backward pass.  Per image i, one launch for the whole batch:
 *   c = cls ? cls[i] : the first argmax of logits[i] (torch.argmax, 分类/test.py:86);
 *   cam[i][y][x] = max(0, sum_k (W[c][k] / (h*w)) * feat[i][y*w+x][k])                              (fp32);
 *   v = cam[i] - min(cam[i]);  v = v / (1e-7f + max(v))             (pytorch-grad-cam scale_cam_image, fp32);
 *   cam_map[i] = 0 outside the box {x0,y0,x1,y1} (end-exclusive, ug_bbox output; NULL = the whole SxS frame), and
 *                cv2.resize(v, (x1-x0, y1-y0), INTER_LINEAR) placed at (x0, y0) inside it (bit-exact against cv2 4.13).
 * cls and boxes may come from outside the library (a plan image's host): an entry whose class is outside [0, ncls) or
 * whose box is not 0 <= x0 < x1 <= S, 0 <= y0 < y1 <= S is rejected: cam[i] and cam_map[i] are zero, status[i] = 1
 * (0 otherwise; status is optional), and nothing is read through that entry.  feat must be 16-byte aligned and C a
 * multiple of 8; h, w <= 32, C <= 2048, S <= 1024. */
typedef struct ug_cam_desc {
  const void* feat;      /* bf16 NHWC [B][h*w][C]: the GoogLeNet inception5b output (h = w = 7, C = 1024) */
  const float* fc_w;     /* fp32 [ncls][C] (the head's weight, unfolded) */
  const float* logits;   /* fp32 [B][ncls]: class = first argmax (torch.argmax, test.py:86), used when cls is NULL */
  const int* cls;        /* optional int32 [B]: explicit target class per image */
  const int* boxes;      /* optional int32 [B][4] {x0,y0,x1,y1} (ug_bbox output, end-exclusive); NULL = the whole SxS frame */
  int* status;           /* optional int32 [B]: 1 = entry rejected (class or box out of range), else 0 */
  float* cam;            /* fp32 [B][h][w]: the Grad-CAM map, ReLU(sum_k W[c][k]/(h*w) * feat[..][k]) */
  float* cam_map;        /* fp32 [B][S][S]: the map normalised and resized into the box, zero outside it */
  int B, h, w, C, ncls, S;
} ug_cam_desc;

/* Source-frame outputs of a pipeline program: each image's mask, ROI box and Grad-CAM map at the image's own size H x W
 * instead of the S x S UNet input frame (S = 224), as a user draws them on the image they read.  Image i is H x W =
 * index[i].H x index[i].W at pixel offset index[i].px_offset (a ragged batch) or Hs x Ws at pixel offset i*Hs*Ws
 * (index NULL).  Per image, one launch for the whole batch:
 *   L = cv2.resize(logits[i], (W, H), INTER_LINEAR) in fp32 (cv2 4.13's scale = in / out, bit-exact);
 *   mask[px + y*W + x] = 1.0f / (1.0f + expf(-L[y][x])) > 0.5f   (the fp32 threshold of the UNet's outc epilogue);
 *   src_boxes[i] = {floor(x0*W/S), floor(y0*H/S), ceil(x1*W/S), ceil(y1*H/S)} for boxes[i] = {x0,y0,x1,y1} (64-bit
 *                  integers): the smallest source-pixel box covering the S-frame box;
 *   with cam: v = cam[i] - min(cam[i]);  v = v / (1e-7f + max(v)) (as ug_cam), and cam_map = cv2.resize(v, (X1-X0,
 *             Y1-Y0), INTER_LINEAR) placed at (X0, Y0) of the source box, zero outside it.
 * When H = W = S the outputs equal the S-frame ones bit for bit (mask, boxes, and ug_cam's cam_map).  The table and the
 * boxes may come from outside the library (a plan image's host): an entry with a negative offset, a side outside
 * [1, 8*S], an extent past capacity_px, or a box that is not 0 <= x0 < x1 <= S, 0 <= y0 < y1 <= S is rejected: nothing
 * is read or written through it, src_boxes[i] = {0,0,0,0} and status[i] = 1 (0 otherwise; status is optional).  The
 * launch geometry depends on B, S and Hs only, never on the table.  logits must be 16-byte aligned, S a multiple of 4
 * and at most 256, h, w <= 32. */
typedef struct ug_source_frame_desc {
  const float* logits;             /* fp32 [B][S][S]: the UNet's segmentation logits (outc output) */
  const int* boxes;                /* int32 [B][4] {x0,y0,x1,y1}, end-exclusive (ug_bbox output) */
  const float* cam;                /* optional fp32 [B][h][w]: ug_cam's raw map; NULL = no CAM map */
  const ug_ragged_image* index;    /* optional device table [B]; NULL = every image is Hs x Ws */
  int* status;                     /* optional int32 [B]: 1 = entry rejected, else 0 */
  unsigned char* mask;             /* u8: image i at mask + px_offset (ragged) or mask + i*Hs*Ws, H*W bytes */
  int* src_boxes;                  /* int32 [B][4]: the box in source pixels, end-exclusive */
  float* cam_map;                  /* fp32, placed like mask; required iff cam is set */
  long long capacity_px;           /* ragged: pixels of mask (and cam_map); unused when index is NULL */
  int B, S, Hs, Ws, h, w;
} ug_source_frame_desc;

enum {
  UG_OP_CONV = 1,
  /* 2 and 10 were the stand-alone im2col packs of round 1 (replaced by UG_OP_STEM); the numbers stay retired */
  UG_OP_POOL = 3,
  UG_OP_LAYERNORM = 4,
  UG_OP_ATTN = 5,
  UG_OP_CHANSTATS = 6,
  UG_OP_GATE = 7,
  UG_OP_BBOX = 8,
  UG_OP_CROPRESIZE = 9,
  UG_OP_HEAD = 11,
  UG_OP_STEM = 12,
  UG_OP_RESIZE = 13,
  UG_OP_WAVELET = 14,
  UG_OP_S2D = 15,
  UG_OP_RESIZE_RAGGED = 16,
  UG_OP_WAVELET_RAGGED = 17,
  UG_OP_CAM = 18,
  UG_OP_SOURCE_FRAME = 19
};

typedef struct ug_op {
  int kind;
  int reserved;
  union {
    ug_conv_desc conv;
    ug_pool_desc pool;
    ug_layernorm_desc ln;
    ug_attn_desc attn;
    ug_chanstats_desc stats;
    ug_gate_desc gate;
    ug_bbox_desc bbox;
    ug_cropresize_desc crop;
    ug_head_desc head;
    ug_stem_desc stem;
    ug_resize_desc resize;
    ug_wavelet_desc wavelet;
    ug_s2d_desc s2d;
    ug_resize_ragged_desc resize_ragged; /* both smaller than ug_conv_desc: sizeof(ug_op) is unchanged */
    ug_wavelet_ragged_desc wavelet_ragged;
    ug_cam_desc cam; /* smaller than ug_conv_desc as well */
    ug_source_frame_desc source_frame; /* and so is this one */
  } u;
} ug_op;

int ug_version(void);
int ug_create(int device, ug_handle* out);
int ug_destroy(ug_handle h);
const char* ug_last_error(ug_handle h);
/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
long long ug_launch_count(ug_handle h);

/* Single ops (validated, tensor maps built per call) — used by the unit parity tests. */
int ug_conv(ug_handle h, const ug_conv_desc* d, void* stream);
int ug_pool(ug_handle h, const ug_pool_desc* d, void* stream);
int ug_layernorm(ug_handle h, const ug_layernorm_desc* d, void* stream);
int ug_attention(ug_handle h, const ug_attn_desc* d, void* stream);
int ug_chanstats(ug_handle h, const ug_chanstats_desc* d, void* stream);
int ug_gate(ug_handle h, const ug_gate_desc* d, void* stream);
int ug_bbox(ug_handle h, const ug_bbox_desc* d, void* stream);
int ug_cropresize(ug_handle h, const ug_cropresize_desc* d, void* stream);
int ug_head(ug_handle h, const ug_head_desc* d, void* stream);
int ug_stem(ug_handle h, const ug_stem_desc* d, void* stream);
int ug_resize_u8(ug_handle h, const ug_resize_desc* d, void* stream);
int ug_wavelet(ug_handle h, const ug_wavelet_desc* d, void* stream);
int ug_s2d_pack(ug_handle h, const ug_s2d_desc* d, void* stream);
int ug_resize_ragged(ug_handle h, const ug_resize_ragged_desc* d, void* stream);
int ug_wavelet_ragged(ug_handle h, const ug_wavelet_ragged_desc* d, void* stream);
int ug_cam(ug_handle h, const ug_cam_desc* d, void* stream);
int ug_source_frame(ug_handle h, const ug_source_frame_desc* d, void* stream);
size_t ug_wavelet_workspace_bytes(int B, int H, int W);
size_t ug_wavelet_ragged_workspace_bytes(int B, long long capacity_px);

/* Programs: a validated op list with tensor maps and launch geometry prepared once; run = launches only. */
int ug_program_create(ug_handle h, const ug_op* ops, int n_ops, ug_program* out);
int ug_program_run(ug_handle h, ug_program p, void* stream);
int ug_program_num_launches(ug_program p);
/* Profiling aid: run with a CUDA event pair around every op, synchronize, and return the device time of each
 * op in milliseconds (ms_per_op has ug_program_num_launches(p) entries). */
int ug_program_run_timed(ug_handle h, ug_program p, void* stream, float* ms_per_op);
int ug_program_destroy(ug_handle h, ug_program p);

/* Host-buffer convenience used for end-to-end timing: H2D copies, run, D2H copies, all on `stream`,
 * then a stream synchronize.  Host pointers should be pinned. */
typedef struct ug_copy {
  void* dst;
  const void* src;
  size_t bytes;
} ug_copy;
int ug_program_run_host(ug_handle h, ug_program p, const ug_copy* h2d, int n_h2d, const ug_copy* d2h, int n_d2h,
                        void* stream);
/* Double-buffered form for back-to-back steps (a serving loop): the H2D copies of this call run on an engine-owned
 * copy stream, so the copy of step i+1 overlaps the kernels of step i; the compute stream then runs the program and
 * enqueues the D2H copies.  Does NOT synchronize: results are valid after the caller synchronizes `stream`.  Two forms:
 *   staged  (stage0 / stage1 non-NULL, each entry at least h2d[i].bytes, caller-owned, alternating per call): the copy
 *           lands in the staging slot and the compute stream moves it into h2d[i].dst (device to device) — one program;
 *   direct  (stage0 == stage1 == NULL): the copy lands in h2d[i].dst itself.  The caller must alternate between TWO
 *           programs with their own input buffers from call to call (call i and call i+2 may share buffers, call i and
 *           call i+1 may not); the extra device-to-device pass of the staged form disappears. */
int ug_program_run_host_pipelined(ug_handle h, ug_program p, const ug_copy* h2d, void* const* stage0,
                                  void* const* stage1, int n_h2d, const ug_copy* d2h, int n_d2h, void* stream);

/* ---- plan images: the net-level entry points (SURVEY.md §8b) -------------------------------------------------------
 * A plan image is a compiled program + its device memory layout + its constant data (BN-folded, packed weights of both
 * networks) as ONE relocatable byte blob, produced once by the Python tooling (`PipelineRunner.export_plan(batch)`,
 * `UNetRunner.export_plan`, `GoogLeNetRunner.export_plan`).  With it a host in any language runs the whole path
 *   UNetTaskAligWeight.forward -> roi.py threshold / bbox / crop / resize -> GoogLeNetClassifier.forward
 * through this C ABI alone (no Python, no CUDA runtime calls of its own):
 *   ug_create -> ug_plan_load -> ug_plan_copy_in("x_in", images) -> ug_plan_run -> ug_plan_copy_out("mask" / "boxes" /
 *   "cls_logits" / "logits" / "u8") -> ug_plan_destroy.     (examples/run_plan.c is exactly this.)
 * Named io buffers of a pipeline plan: "x_in" f32 [B,3,224,224] (or "src_u8" u8 [B,Hs,Ws,3] for plans with the device
 * front-end), "logits" f32 [B,1,224,224], "mask" u8 [B,224,224], "boxes" i32 [B,4], "u8" u8 [B,224,224,3] (the ROI
 * crops), "cls_logits" f32 [B,6].  A ragged plan (export_plan(B, source="ragged", capacity=P)) takes packed sources
 * instead: "src_u8" u8 [P*3] (images back to back, HWC), "src_index" ug_ragged_image [B] and reports "src_status"
 * i32 [B] (1 = the table entry was rejected and the image's outputs are those of a zero input).  A plan exported with
 * cam=True (export_plan(B, ..., cam=True)) also reports the Grad-CAM of each image's predicted class (ug_cam_desc):
 * "cam" f32 [B,7,7] and "cam_map" f32 [B,224,224] (the map in the UNet input frame, inside the ROI box).  A plan
 * exported with source_frame=True (a plan with a uint8 or ragged source) also reports the outputs at each image's own
 * size (ug_source_frame_desc): "src_mask" u8 [B,Hs,Ws] (ragged: [P], image i at px_offset), "src_boxes" i32 [B,4]
 * and, with cam=True, "src_cam_map" f32 [B,Hs,Ws] (ragged: [P]). */
typedef struct ug_plan_s* ug_plan;
/* Parses the image (host memory, may be freed afterwards), allocates ONE device arena for every buffer of the plan
 * (ug_plan_device_bytes), uploads the constants, relocates the op list and prepares the program. */
int ug_plan_load(ug_handle h, const void* image, size_t image_bytes, ug_plan* out);
int ug_plan_num_io(ug_plan p);
const char* ug_plan_io_name(ug_plan p, int i);
/* Device pointer and size of a named io buffer (UG_EINVAL if the plan has no such buffer). */
int ug_plan_io(ug_plan p, const char* name, void** dev_ptr, size_t* bytes);
size_t ug_plan_device_bytes(ug_plan p);
/* The prepared program of the plan (for ug_program_run_host / _pipelined / _timed). */
ug_program ug_plan_program(ug_plan p);
/* Host -> named buffer (asynchronous on `stream`) / named buffer -> host (synchronizes `stream`). */
int ug_plan_copy_in(ug_handle h, ug_plan p, const char* name, const void* host, size_t bytes, void* stream);
int ug_plan_copy_out(ug_handle h, ug_plan p, const char* name, void* host, size_t bytes, void* stream);
int ug_plan_run(ug_handle h, ug_plan p, void* stream);
int ug_plan_destroy(ug_handle h, ug_plan p);

#ifdef __cplusplus
}
#endif
#endif /* UGNET_H_ */
