/* libmitb -- C ABI of the B200-native detect -> OCR -> inpaint hot path.
 *
 * Drop-in boundary for manga-image-translator's three dense-inference plugins.  Every entry point replaces the
 * torch call made by the reference at the cited line (paths relative to manga_translator/):
 *
 *   mitb_dbnet_forward[_u8]  <- det_batch_forward_default: MODEL(batch); db.sigmoid()   detection/dbnet_convnext.py:499-509
 *   mitb_ocr_forward[_u8]    <- OCR.decode up to the host loop: backbone, encoders, heads,
 *                               log_softmax + max, colour clamp                           ocr/model_48px_ctc.py:447-463
 *   mitb_lama_forward        <- LamaFourier.__call__ (inpaint_only): MPE embed, generator,
 *                               pred*mask+(1-mask)*img                                    inpainting/inpainting_lama_mpe.py:713-726
 *   mitb_*_load / _unload    <- the plugins' _load/_unload (torch.load + load_state_dict)  dbnet_convnext.py:527-539,
 *                               model_48px_ctc.py:38-60, inpainting_lama_mpe.py:46-51,131-136,818-825
 *
 * Conventions: plain C, no exceptions cross the boundary.  Every function returns 0 on success, non-zero on
 * failure with the message available from mitb_last_error().  All data pointers are DEVICE pointers on the
 * context's GPU (fp32 NCHW like the reference tensors) unless the name says _u8/host; `stream` is a cudaStream_t
 * (NULL = default stream) and calls are asynchronous on it.  A context is bound to one GPU and is not re-entrant.
 * There is no CPU fallback: without a CUDA device mitb_create fails.
 */
#ifndef MITB_H
#define MITB_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mitb_ctx mitb_ctx;

/* One named fp32 tensor of a PyTorch state_dict, resident on the device (contiguous, row-major). */
typedef struct {
  const char* name;      /* state_dict key, e.g. "backbone.stem.0.weight" */
  const float* data;     /* device pointer */
  int32_t ndim;          /* 0..4 */
  int64_t shape[4];
} mitb_tensor;

int mitb_create(int device_ordinal, mitb_ctx** out);
void mitb_destroy(mitb_ctx* ctx);
const char* mitb_last_error(const mitb_ctx* ctx);      /* valid until the next call on ctx; ctx may be NULL */
const char* mitb_version(void);
long long mitb_launch_count(const mitb_ctx* ctx);      /* kernels launched by this context so far */
size_t mitb_workspace_bytes(const mitb_ctx* ctx);      /* current activation workspace size */

/* Process-wide switch between the tcgen05 (bf16x3 split, ~1e-5 relative) and the exact-fp32 SIMT convolution kernels.
 * Default on.  The SIMT kernels are the parity anchor of the tensor-core path (tests run both). */
int mitb_set_tensor_cores(int on);
/* LaMa FFC layer implementation (process-wide): 0 = generic planar path (any size), 1 = fused NHWC path (operand-fused GEMMs +
 * channel-vectorised FFT; sizes whose bottleneck h/8, w/8 are {2,3,5}-smooth) when the page is large enough that no layer
 * needs split-K (default), 2 = fused path whenever it is capable (tests). */
int mitb_set_ffc_mode(int mode);
/* Process-wide: LaMa's decoder (three transposed convs + the 7x7 output conv) computes only the tiles from which a hole pixel of
 * the final blend `pred*mask + (1-mask)*img` (inpainting_lama_mpe.py:726) is reachable; every used pixel is bit-identical to the dense
 * computation (on by default; 0 = dense, also MITB_DENSE_TAIL=1). */
int mitb_set_sparse_decoder(int on);

/* Per-launch CUDA-event timing aggregated per kernel class (for bench.py's roofline block). report() synchronises the
 * recorded events, clears them and returns a JSON object {"class": {"launches","ms","flops","bytes"}, ...} valid until
 * the next call. */
int mitb_profile_enable(mitb_ctx* ctx, int on);
const char* mitb_profile_report(mitb_ctx* ctx);

/* ---- DBNet-ConvNeXt text detector (state_dict keys of DBNetConvNext, dbnet_convnext.py:450-472) ---- */
int mitb_dbnet_load(mitb_ctx* ctx, const mitb_tensor* weights, int n_weights);
int mitb_dbnet_unload(mitb_ctx* ctx);
/* x: [n,3,h,w] already normalised (u8/127.5-1), h and w multiples of 128 (the reference pads to 256).
 * db: [n,2,h,w] = sigmoid(DBHead output) (channel 1 is sigmoid applied twice, as the reference does);
 * mask: [n,1,h/2,w/2]. */
int mitb_dbnet_forward(mitb_ctx* ctx, const float* x, int n, int h, int w, float* db, float* mask, void* stream);
/* Same, input uint8 NHWC [n,h,w,3] on the device; the u8/127.5-1 normalisation is fused into the first kernel. */
int mitb_dbnet_forward_u8(mitb_ctx* ctx, const uint8_t* img, int n, int h, int w, float* db, float* mask, void* stream);

/* ---- 48px ResNet+Transformer CTC recogniser (state_dict keys of OCR, model_48px_ctc.py:425-436) ---- */
int mitb_ocr_load(mitb_ctx* ctx, const mitb_tensor* weights, int n_weights);
int mitb_ocr_unload(mitb_ctx* ctx);
int mitb_ocr_timesteps(int wp);                         /* T = floor(floor(wp/2)/2) - 1 */
/* x: [n,3,48,wp] normalised ((u8-127.5)/127.5).  Outputs per timestep, T = mitb_ocr_timesteps(wp):
 * argmax [n,T] int32, logprob [n,T] (log-softmax value at the argmax), colors [n,T,6] clamped to [0,1].
 * The [n,T,V] logits are never materialised. */
int mitb_ocr_forward(mitb_ctx* ctx, const float* x, int n, int wp, int32_t* argmax, float* logprob, float* colors,
                     void* stream);
int mitb_ocr_forward_u8(mitb_ctx* ctx, const uint8_t* img /*[n,48,wp,3]*/, int n, int wp, int32_t* argmax,
                        float* logprob, float* colors, void* stream);

/* ---- LaMa FFC inpainter, MPE (9 blocks + str_state_dict) or large (18 blocks) ----
 * weights: generator keys "model.*" plus, for MPE, "mpe.rel_pos_emb.weight", "mpe.direct_emb.weight",
 * "mpe.alpha5", "mpe.alpha6" (the str_state_dict keys prefixed with "mpe."). */
int mitb_lama_load(mitb_ctx* ctx, const mitb_tensor* weights, int n_weights);
int mitb_lama_unload(mitb_ctx* ctx);
/* img [n,3,h,w] in [0,1] (pre-masked or not: the generator multiplies by 1-mask itself), mask [n,1,h,w] in {0,1},
 * h and w multiples of 8; rel_pos int32 [n,h,w] in [0,127] and direct int32 [n,h,w,4] in {0,1} are the MPE tables
 * (NULL for the large model); out [n,3,h,w] = pred*mask + (1-mask)*img. */
int mitb_lama_forward(mitb_ctx* ctx, const float* img, const float* mask, const int32_t* rel_pos,
                      const int32_t* direct, int n, int h, int w, float* out, void* stream);

/* Same, with the MPE tables at the 256x256 working resolution of load_masked_position_encoding (:751-815): rel_pos256
 * [n,256,256], direct256 [n,256,256,4]; the INTER_NEAREST upsampling and the zeroing outside the hole (:807-813) happen
 * inside the kernel that adds the embeddings. */
int mitb_lama_forward_mpe256(mitb_ctx* ctx, const float* img, const float* mask, const int32_t* rel_pos256,
                             const int32_t* direct256, int n, int h, int w, float* out, void* stream);

/* uint8 entry covering the whole device part of LamaMPEInpainter._infer (inpainting_lama_mpe.py:82-117) for one image:
 * img uint8 [h,w,3] and mask uint8 [h,w] on the device (already resized to the network resolution, multiples of 8);
 * normalisation (/255), mask binarisation (>=0.5), pre-masking, the network, pred*mask+(1-mask)*img, (x*255) truncation to
 * uint8 and -- when composite != 0 -- `ans = inpainted*m0 + img*(1-m0)` with m0 = (mask >= 127) all run in kernels.
 * rel_pos256/direct256: the 256x256 MPE tables (NULL for the large model). out: uint8 [h,w,3]. */
int mitb_lama_infer_u8(mitb_ctx* ctx, const uint8_t* img, const uint8_t* mask, const int32_t* rel_pos256,
                       const int32_t* direct256, int h, int w, int composite, uint8_t* out, void* stream);

/* ---- standalone operators (parity tests and micro-benchmarks; same kernels the networks use) ---- */
/* General conv through the implicit-GEMM kernel.  x [n,cin,h,w], wt PyTorch layout [cout,cin,kh,kw], y [n,cout,ho,wo]
 * (all NCHW device fp32).  pad_mode 0 zero / 1 reflect; act 0 none,1 relu,2 gelu(erf),3 silu,4 sigmoid.
 * bias / in_scale / in_shift may be NULL; in_relu applies relu(x*in_scale+in_shift) before the conv. */
int mitb_op_conv2d(mitb_ctx* ctx, const float* x, int n, int cin, int h, int w, const float* wt, int cout, int kh,
                   int kw, int stride_y, int stride_x, int pad_y, int pad_x, int pad_mode, const float* bias, int act,
                   const float* in_scale, const float* in_shift, int in_relu, float* y, void* stream);
/* ConvTranspose2d, stride 2: (k=2,p=0,op=0), (k=4,p=1,op=0) or (k=3,p=1,op=1).  wt [cin,cout,k,k]. */
int mitb_op_conv_transpose2d(mitb_ctx* ctx, const float* x, int n, int cin, int h, int w, const float* wt, int cout,
                             int k, int pad, int out_pad, const float* bias, int act, float* y, void* stream);
/* depthwise 7x7 (pad 3, bias) + LayerNorm over C (eps), NCHW in/out. */
int mitb_op_dwconv7_ln(mitb_ctx* ctx, const float* x, int n, int c, int h, int w, const float* wdw, const float* bdw,
                       const float* lnw, const float* lnb, float eps, float* y, void* stream);
/* LayerNorm over the last dim of [rows, c]. */
int mitb_op_layernorm(mitb_ctx* ctx, const float* x, int rows, int c, const float* w, const float* b, float eps,
                      float* y, void* stream);
/* torch.fft.rfftn / irfftn over (h,w), norm='ortho', planar [c,h,w] <-> [2c,h,w/2+1] (re/im interleaved per channel). */
int mitb_op_rfft2(mitb_ctx* ctx, const float* x, int c, int h, int w, float* spec, void* stream);
int mitb_op_irfft2(mitb_ctx* ctx, const float* spec, int c, int h, int w, float* y, void* stream);
/* Same transforms on NHWC tensors (the layout of the fused FFC path): x [n,h,w,c] -> spec [n,h,w/2+1,2c] (c0_re,c0_im,c1_re,...);
 * irfft adds `add` [n,h,w,c] when non-NULL (the x + fu(x) residual, inpainting_lama_mpe.py:305).  h, w {2,3,5}-smooth, c even. */
int mitb_op_rfft2_nhwc(mitb_ctx* ctx, const float* x, int n, int h, int w, int c, float* spec, void* stream);
int mitb_op_irfft2_nhwc(mitb_ctx* ctx, const float* spec, const float* add, int n, int h, int w, int c, float* y, void* stream);
/* Multi-head attention core: qk [n*t, 2*d] (q then k, already projected), v [n*t, d] -> out [n*t, d], d = heads * head_dim, no mask.
 * Any alignment.  Any t for head_dim <= 64 (the OCR: 8 x 40, t <= 2048); for head_dim > 64 only t with
 * 4 * (2 * t * (head_dim + 1) + 8 * t + 8 * head_dim) <= 200 KB (K / V of a head held whole in shared memory), else an error. */
int mitb_op_attention(mitb_ctx* ctx, const float* qk, const float* v, int n, int t, int heads, int head_dim,
                      float* out, void* stream);
/* LamaFourier.load_masked_position_encoding at its 256x256 working resolution (inpainting_lama_mpe.py:763-803): small = the
 * INTER_AREA-reduced uint8 mask [n,256,256] (hole where != 0) -> rel_pos int32 [n,256,256] in [0,127], direct int32 [n,256,256,4]. */
int mitb_op_mpe_tables(mitb_ctx* ctx, const uint8_t* small, int n, int32_t* rel_pos, int32_t* direct, void* stream);
/* cv2.bilateralFilter(img, 17, 80, 80) on a uint8 HWC3 device image (detector pre-filter, dbnet_convnext.py:549). */
int mitb_op_bilateral17(mitb_ctx* ctx, const uint8_t* img, int h, int w, uint8_t* out, void* stream);

/* Text-line crops on the device (SURVEY 8f N2 / row O3): for each of the n lines of an OCR chunk,
 * cv2.warpPerspective(page[y1:y2, x1:x2], M, (w, h)) [+ cv2.rotate(ROTATE_90_COUNTERCLOCKWISE) for vertical lines] of
 * Quadrilateral.get_transformed_region (utils/generic.py:445-481), written into the zero-padded chunk canvas
 * uint8 [n, canvas_h, canvas_w, 3] of Model48pxCTCOCR._infer (ocr/model_48px_ctc.py:86-92).  Bit-exact with OpenCV (INTER_LINEAR,
 * BORDER_CONSTANT 0).  page: uint8 [h, w, 3] on the device.  lines: device double [n][16] = { Minv[9] (inverse of the homography the
 * host solved with cv2.findHomography, row major), x1, y1, crop_w, crop_h, out_w, out_h (before the rotation), rot (0 / 1) }. */
int mitb_op_warp_lines_u8(mitb_ctx* ctx, const uint8_t* page, int h, int w, const double* lines, int n, uint8_t* canvas, int canvas_h,
                          int canvas_w, void* stream);
/* Greedy CTC collapse of decode_ctc_top1 (ocr/model_48px_ctc.py:466-478, row O8): per line keep step t iff argmax[t] != 0 (blank) and
 * argmax[t] != argmax[t-1]; counts int32 [n]; the kept steps, their character ids, log-probabilities and colours are compacted to the
 * front of steps / chars int32 [n,t], logprob_out [n,t], colors_out [n,t,6] (the last two may be NULL). */
int mitb_op_ctc_collapse(mitb_ctx* ctx, const int32_t* argmax, const float* logprob, const float* colors, int n, int t, int32_t* counts,
                         int32_t* steps, int32_t* chars, float* logprob_out, float* colors_out, void* stream);

/* SURVEY 8f N3: `quadrilateral_can_merge_region` (utils/generic.py:653-698) for every pair of text lines - the O(n^2) part of the OCR
 * direction graph (ocr/common.py:12-39) and of textline_merge (textline_merge/__init__.py:110-126).  quads: device double [n][16] =
 * corners (8), AABB x, y, w, h, font_size, aspect_ratio, angle, flags (bit 0 approximately axis aligned, bit 1 convex).
 * adj: uint8 [n][n], symmetric: 1 mergeable, 0 not, 2 undecided (a non-convex quad: the caller evaluates that pair itself). */
int mitb_op_textline_pairs(mitb_ctx* ctx, const double* quads, int n, double ratio, double discard_connection_gap, double char_gap_tolerance,
                           double char_gap_tolerance2, double font_size_ratio_tol, double aspect_ratio_tol, uint8_t* adj, void* stream);

/* ---- mask refinement (SURVEY 8f N1; manga_translator/mask_refinement/__init__.py:9-31, text_mask_utils.py:64-190) ---- */
/* cv2.resize(src, (dw, dh), interpolation=INTER_LINEAR) for uint8 [sh,sw,channels] (channels 1 or 3), bit-exact; binarize != 0
 * additionally maps every non-zero result to 255 (`mask[mask > 0] = 255`, __init__.py:18,28). */
int mitb_op_resize_linear_u8(mitb_ctx* ctx, const uint8_t* src, int sh, int sw, int channels, uint8_t* dst, int dh, int dw, int binarize, void* stream);
/* cv2.rectangle(mask, (x, y), (x + w, y + h), 0, 1) for n rectangles (rects int32 [n][4] = x, y, w, h; text_mask_utils.py:99-100). */
int mitb_op_cut_rects(mitb_ctx* ctx, uint8_t* mask, int h, int w, const int32_t* rects, int n, void* stream);
/* cv2.connectedComponentsWithStats(mask) (8-connectivity): labels int32 [h*w] = component id in [0, ncomp) or -1 for background (ids are
 * in no particular order - the reference's use of them is order independent), stats int32 [cap][5] = {x0, y0, x1, y1, area},
 * ncomp int32 [1] (components beyond `cap` get label -1; the caller checks ncomp <= cap).  scratch: int32 [2*h*w]. */
int mitb_op_cc_label(mitb_ctx* ctx, const uint8_t* mask, int h, int w, int32_t* labels, int32_t* stats, int32_t* ncomp, int cap, int32_t* scratch,
                     void* stream);
/* owner_map[i] = owner[labels[i]] (text line owning the pixel's component, -1: none): all textline_ccs of complete_mask in one map. */
int mitb_op_owner_map(mitb_ctx* ctx, const int32_t* labels, const int32_t* owner, int n, int32_t* owner_map, void* stream);
/* refine_mask (text_mask_utils.py:71-94) for all text lines of a page at once: DenseCRF2D with unary_from_softmax of the line's
 * component mask, addPairwiseGaussian(sxy_g, w_g), addPairwiseBilateral(sxy_b, srgb, w_b) (DIAG_KERNEL, NO_NORMALIZATION), `iters`
 * mean-field iterations, argmax.  lines2 / lines5: int32 [nlines][8] = {x, y, w, h (region in the working image), first pixel of the
 * region's segment, first slot and capacity (power of two, >= 2 (d+1) w h) of its hash-table segment, 0} for the d = 2 and d = 5
 * lattices; img uint8 [h,w,3] (the bilateral-filtered working image); refined uint8 [npix] (255: text).  err int32 [1]: non-zero if a
 * lattice key left the packed range or a table overflowed.  work: device scratch of mitb_op_crf_workspace bytes. */
int mitb_op_crf_workspace(long long npix, long long nslots2, long long nslots5, unsigned long long* bytes);
int mitb_op_dense_crf(mitb_ctx* ctx, const int32_t* lines2, const int32_t* lines5, int nlines, const uint8_t* img, const int32_t* owner_map, int img_w,
                      int max_pix, int max_cap2, int max_cap5, long long npix, long long nslots2, long long nslots5, int iters, float sxy_g,
                      float w_g, float sxy_b, float srgb, float w_b, float u_on, void* work, uint8_t* refined, int32_t* err, void* stream);
/* Per line: cc = refined inside rect1, (owner_map == line) elsewhere; cv2.dilate(cc[rect2], ellipse) OR-ed into final_mask
 * (text_mask_utils.py:183-186).  lines int32 [nlines][12] = {x1,y1,w1,h1, x2,y2,w2,h2, first pixel of the refined segment, offset of
 * the line's structuring element in `se`, its size, 0}. */
int mitb_op_dilate_lines(mitb_ctx* ctx, const int32_t* lines, int nlines, int max_pix2, const int32_t* owner_map, const uint8_t* refined,
                         const uint8_t* se, int img_w, uint8_t* final_mask, void* stream);
/* cv2.dilate(src, se) for a uint8 image and a ksize x ksize structuring element (anchor at the centre). */
int mitb_op_dilate_se(mitb_ctx* ctx, const uint8_t* src, int h, int w, const uint8_t* se, int ksize, uint8_t* dst, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MITB_H */
