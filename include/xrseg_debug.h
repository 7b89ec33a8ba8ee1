/*
 * xrseg_debug.h -- parity / probe entry points exported ONLY by libxrseg_debug.so (the same sources as libxrseg.so built
 * with -DXRSEG_DEBUG_API; xr_image_segmentation_b200/csrc/Makefile).  libxrseg_debug.so also exports everything in
 * xrseg.h, so a test creates its runner and calls these hooks in ONE library.  Nothing here is product surface: these
 * functions feed caller-made tensors to single kernels, fetch intermediate activations, or emulate data movement on the
 * host for CPU tests of the index math.
 */
#ifndef XRSEG_DEBUG_H_
#define XRSEG_DEBUG_H_

#include "xrseg.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Copy a named intermediate activation of the last run to host as f32 NCHW [n,C,H,W].
 * names: "p3","p4","p5","box_logits.i","cls_logits.i","coefs.i" (i = 0..2),"protos","input", every layer name, and the
 * outputs of the copy / max-pool launches: "b9.pool" (the three chained SPPF max-pools), "up.13" / "up.16" (the nearest
 * x2 upsamples feeding n13 / n16).
 * A run of batch > micro_batch computes its frames in chunks of micro_batch that reuse one activation arena, so only the
 * LAST chunk is resident: the fetched frames are (ceil(batch / micro_batch) - 1) * micro_batch .. batch - 1, and
 * shape4[0] = n is their count.  A zero-capacity call reports the shape and returns XRSEG_ERR_CAPACITY. */
int xrseg_debug_fetch(xrseg_runner* r, const char* name, float* dst, size_t cap_floats, int64_t* shape4);
/* Same as xrseg_debug_fetch, for `count` frames starting at frame `first` of the resident chunk (first = 0 is its first
 * frame; count = -1: to its end).  At large batches a whole layer is gigabytes of fp32: a test that checks a few frames
 * copies only those.  Frames outside the resident chunk: XRSEG_ERR_INVALID. */
int xrseg_debug_fetch_frames(xrseg_runner* r, const char* name, int first, int count, float* dst, size_t cap_floats,
                             int64_t* shape4);
/* The launch list of the last run's resident (last) chunk, in launch order: per launch the CTAs of its grid, its work items
 * and, for a convolution on the tcgen05 engine, its mode (conv_umma.cuh MODE_*; -1 for every other launch).  grid and items
 * are 0 for the stem, whose kernel is chosen when it is launched.  names: cap * 32 bytes (may be NULL).  Returns the number
 * of launches, XRSEG_ERR_CAPACITY when cap is smaller. */
int xrseg_debug_launches(xrseg_runner* r, int* grid, int* items, int* mode, char* names, int cap);
/* Run ONLY the post-processing stage on caller-provided fp32 head tensors (the oracle's own tensors):
 * box_logits [batch,A,64], cls_logits [batch,A,nc] (nc = the runner's xrseg_num_classes), coefs [batch,A,32],
 * protos [batch,32,160*160]. */
int xrseg_debug_post(xrseg_runner* r, const float* box_logits, const float* cls_logits, const float* coefs,
                     const float* protos, int batch);
/* Same tensors through the PRODUCT kernels: rounded to fp16 on the device (prototypes re-laid out NHWC like the network's),
 * then the streaming decode filter, NMS and the mma.sync mask assembly of the per-frame path (tools/bench_post.py:
 * BASELINE.json configs[4], the post-processing stress shape).  XRSEG_MASK_UPSAMPLE_640 then reads these prototypes; after
 * xrseg_debug_post (fp32, planar) it returns XRSEG_ERR_STATE. */
int xrseg_debug_post_f16(xrseg_runner* r, const float* box_logits, const float* cls_logits, const float* coefs,
                         const float* protos, int batch);
/* Per-launch CUDA-event times of the last xrseg_debug_post* call made with XRSEG_DBG_TIME=1 in the environment
 * (bench.py --config 4): ms[i], algorithmic bytes[i], names[i*32].  Returns the number of launches. */
int xrseg_debug_post_timings(xrseg_runner* r, float* ms, double* bytes, char* names, int cap);
/* NMS alone on caller-provided corners [batch,A,4] + scores [batch,A]; results through xrseg_keep_indices. */
int xrseg_debug_nms(xrseg_runner* r, const float* corners, const float* scores, int batch, int num_anchors);
/* Threshold + crop of caller-provided mask probabilities f32 [n,160,160] with caller boxes (C# convention
 * boxes, 4 floats each) -- the bit-exact leg of IEMasker. */
int xrseg_debug_mask_threshold(xrseg_runner* r, const float* probs, const float* boxes, int n, int image_w,
                               int image_h, float thr, uint8_t* out);
/* One convolution through the selected engine: x f32 NCHW [b,cin,h,w], w f32 [cout,cin/g,k,k] (or
 * [cin,cout,k,k] when transposed), optional residual f32 NCHW; y f32 NCHW out. */
int xrseg_debug_conv(int device, int impl, const float* x, int b, int cin, int h, int w, const float* wgt,
                     const float* bias, int cout, int k, int stride, int groups, int act, int transposed,
                     const float* residual, float* y, int variant);
/* The fused Bottleneck kernel (Conv3x3+SiLU -> Conv3x3+SiLU (+ x), graph chains X.m0.cv1 / X.m0.cv2 of the C3k2 blocks,
 * SURVEY.md Appendix A) on caller tensors: x f32 NCHW [b,c1,h,w], w1 [cm,c1,3,3], w2 [c2,cm,3,3]; y f32 NCHW out.
 * Channel triples: 16-8-16 and 32-16-32 (after padding). */
int xrseg_debug_bottleneck(int device, const float* x, int b, int c1, int h, int w, const float* w1, const float* b1,
                           int cm, const float* w2, const float* b2, int c2, int residual, float* y);
/* Host-only: weight packing of the fused Bottleneck kernel into mma.sync B-fragment order (CPU layout tests). */
int xrseg_debug_pack_bneck(const float* w, int cin, int cout, int C, int N, int taps, uint32_t* out, size_t cap_words);
/* Host-side emulation of the UMMA conv kernel's data movement (slot mapping, weight packing, tap shifts)
 * in fp32 -- used by CPU tests to validate index math without a GPU.  NOT a product path. */
int xrseg_debug_emulate_conv(const float* x, int b, int cin, int h, int w, const float* wgt, const float* bias,
                             int cout, int k, int stride, int act, int transposed, const float* residual,
                             float* y, int variant);

/* The C2PSA attention kernel alone (graph chains 160-168: Q^T K * 0.17678, softmax over keys, V A^T) on caller tensors:
 * qkv f32 [b, n, heads*128] (per token and head: 32 query | 32 key | 64 value channels), out f32 [b, n, heads*64]. */
int xrseg_debug_attention(int device, const float* qkv, int b, int n, int heads, float* out, const float* pe_w, const float* pe_b,
                          int map_w);   /* pe_w [heads*64][3][3] + pe_b [heads*64]: fused positional encoding (NULL: attention only) */

#ifdef __cplusplus
}
#endif
#endif /* XRSEG_DEBUG_H_ */
