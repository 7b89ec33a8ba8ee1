/*
 * xrseg.h -- C ABI of libxrseg.so, the B200-native (sm_100a) replacement for the per-frame
 * YOLO11-seg hot path of netlab-dgist/xr-image-segmentation.
 *
 * The reference has no native boundary today (no DllImport anywhere); its hot path talks to the
 * Unity Inference Engine `Worker` / `Tensor` API from
 *   Assets/Scripts/InferenceEngine/IEExecutor.cs   (IEE)
 *   Assets/Scripts/InferenceEngine/IEBoxer.cs      (IEB)
 *   Assets/Scripts/InferenceEngine/IEMasker.cs     (IEM)
 * Each entry point below names the reference call it replaces (file:line).  A C# P/Invoke stub and the
 * ctypes binding are shown in INTEGRATION.md.
 *
 * Conventions: plain C types only; every call returns XRSEG_OK (0) or a negative xrseg_status; no
 * exceptions, no callbacks; one thread per runner at a time; one runner per GPU.  There is no CPU
 * fallback: without a CUDA device (or with a non-sm_100 device) xrseg_create fails.
 */
#ifndef XRSEG_H_
#define XRSEG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XRSEG_ABI_VERSION 2

typedef enum xrseg_status {
  XRSEG_OK = 0,
  XRSEG_ERR_INVALID = -1,      /* bad argument */
  XRSEG_ERR_CUDA = -2,         /* CUDA runtime error, see xrseg_last_error */
  XRSEG_ERR_NO_DEVICE = -3,    /* no usable sm_100 device (there is no CPU fallback) */
  XRSEG_ERR_WEIGHTS = -4,      /* weight pack does not match the requested topology */
  XRSEG_ERR_STATE = -5,        /* call not valid in the current runner state (e.g. peek before schedule) */
  XRSEG_ERR_NO_DETECTIONS = -6,/* run finished with N == 0 (the reference's Error state, IEE:453-454) */
  XRSEG_ERR_CAPACITY = -7      /* destination buffer too small, or (from xrseg_poll / xrseg_wait / the first accessor of a
                                  finished run) the run hit max_candidates / max_det: results are truncated, see
                                  xrseg_overflow */
} xrseg_status;

typedef enum xrseg_pixel_format {
  XRSEG_FMT_RGB8 = 0,          /* 3 bytes per pixel, top row first */
  XRSEG_FMT_RGBA8 = 1,         /* 4 bytes per pixel, alpha ignored (Quest passthrough WebCamTexture) */
  /* Row order.  By default the FIRST row in memory is the TOP row of the picture (what the Python mirror's ToTensor and
   * every test feed).  OR this flag into `fmt` when the buffer is bottom-up, i.e. memory row 0 is the BOTTOM of the
   * picture -- Unity's Texture2D.GetPixels32 / WebCamTexture.GetPixels32 / GetRawTextureData order (texture origin
   * bottom-left), which TextureConverter.ToTensor (IEE:370) turns into a top-first tensor internally.  The stem and the
   * resample kernel then read image row y from memory row h-1-y; nothing is copied. */
  XRSEG_FMT_BOTTOM_UP = 0x100
} xrseg_pixel_format;

typedef enum xrseg_resize_mode {
  XRSEG_RESIZE_STRETCH = 0,    /* what TextureConverter.ToTensor(tex,640,640,3) does (IEE:370) */
  XRSEG_RESIZE_LETTERBOX = 1   /* extension: aspect-preserving, pad 114 (BASELINE.json config 4) */
} xrseg_resize_mode;

typedef enum xrseg_dtype { XRSEG_F32 = 0, XRSEG_I32 = 1, XRSEG_F16 = 2, XRSEG_U8 = 3 } xrseg_dtype;

/* Conv engine selection (debug / parity only; the product default is XRSEG_CONV_UMMA). */
typedef enum xrseg_conv_impl {
  XRSEG_CONV_UMMA = 0,         /* tcgen05/TMEM implicit GEMM */
  XRSEG_CONV_DIRECT = 1        /* plain CUDA-core direct convolution (on-GPU cross-check) */
} xrseg_conv_impl;

typedef struct xrseg_runner xrseg_runner;

/* ↔ the serialized inspector fields of IEExecutor (IEE:27-44) plus the thresholds baked into the asset
 * by IEModelEditorConverter.cs:76 (decoded: iou 0.43, score 0.301) and IEE:32 (_confidenceThreshold 0.5). */
typedef struct xrseg_config {
  uint32_t struct_size;        /* = sizeof(xrseg_config) */
  int32_t device;              /* CUDA device ordinal */
  int32_t max_batch;           /* frames per schedule call (1 = the reference's behaviour) */
  int32_t model_scale;         /* 'n' or 's' */
  const void* weights;         /* host memory: the sample's .sentis asset bytes (yolo11n-seg-sentis.sentis, loaded like
                                  ModelLoader.Load, IEE:382) or an XRSW weight pack (weights.py) */
  size_t weights_bytes;
  float iou_threshold;         /* 0 -> 0.43 (or the value baked into a .sentis asset) */
  float score_threshold;       /* 0 -> 0.301 (ditto) */
  float mask_threshold;        /* 0 -> 0.5 (IEE:32 _confidenceThreshold); negative -> exactly 0 */
  /* DEVIATION from the reference, which runs NonMaxSuppression unlimited (maxOutputBoxesPerClass = -1,
   * IEModelEditorConverter.cs:76): device buffers are sized by these two caps.  A run that exceeds either is NOT silently
   * truncated: xrseg_poll / xrseg_wait (or the first accessor) return XRSEG_ERR_CAPACITY once, xrseg_overflow() tells
   * which cap was hit, and the truncated results stay readable.  max_candidates = 8400 and max_det = 8400 reproduce the
   * unlimited behaviour exactly (at 8.9 MB of IoU bitmask and 860 MB of mask probabilities per frame of max_batch). */
  int32_t max_det;             /* per-frame cap on kept detections, 0 -> 300 */
  int32_t max_candidates;      /* per-frame cap on score-filtered candidates entering NMS, 0 -> 2048 */
  int32_t resize_mode;         /* xrseg_resize_mode */
  int32_t conv_impl;           /* xrseg_conv_impl */
  int32_t use_cuda_graph;      /* 1 = replay the captured pipeline (default 1) */
  int32_t micro_batch;         /* frames pushed through the network per pass, 0 -> auto */
  int32_t num_classes;         /* classes of the model (1..1024): 0 -> taken from the weights; any other value must equal
                                  the weights' count, else xrseg_create fails with XRSEG_ERR_WEIGHTS */
  int32_t reserved[7];
} xrseg_config;

/* Borrowed view of an output tensor: valid until the next xrseg_schedule (↔ Worker.PeekOutput, IEE:426). */
typedef struct xrseg_tensor_view {
  const void* device_ptr;      /* device memory, rows compacted over the batch in frame order */
  int32_t dtype;               /* xrseg_dtype */
  int32_t rank;
  int64_t shape[4];            /* shape[0] = total detections over the batch */
} xrseg_tensor_view;

/* ↔ struct BoundingBox (IEB:6-15); ClassName/Label are the label id, resolved by the host with
 * xrseg_class_name semantics (IEB:183-188). */
typedef struct xrseg_box {
  float center_x, center_y, width, height;
  int32_t label_id;
  int32_t frame;               /* frame index inside the batch */
} xrseg_box;

typedef enum xrseg_box_convention {
  XRSEG_BOX_PARSEBOXES = 0,    /* IEExecutor.ParseBoxes, IEE:529-559: centred, Y-up, cap 50 */
  XRSEG_BOX_DRAWBOXES = 1,     /* IEBoxer.DrawBoxes, IEB:37-81: centred, Y-down, cap 200 */
  XRSEG_BOX_RAW = 2            /* cx,cy,w,h in 640-px input space (output_0 rows) */
} xrseg_box_convention;

typedef enum xrseg_mask_mode {
  XRSEG_MASK_REFERENCE_160 = 0,/* IEMasker.DrawMask / DrawSingleMask (IEM:98-113,167-185): prob > thr &&
                                  PixelInBoundingBox, texture row order (posY = 159 - y), u8 0/1 [n,160,160] */
  XRSEG_MASK_CROP_160 = 1,     /* extension: geometric crop in image row order, u8 [n,160,160] */
  XRSEG_MASK_UPSAMPLE_640 = 2, /* extension: bilinear 160->640 of the logits, crop, threshold, u8 [n,640,640] */
  XRSEG_MASK_BITS_160 = 3      /* extension: XRSEG_MASK_CROP_160 bit-packed, 32 pixels per u32, [n,160,5] */
} xrseg_mask_mode;

typedef struct xrseg_mask_params {
  uint32_t struct_size;
  int32_t mode;                /* xrseg_mask_mode */
  int32_t box_convention;      /* for MODE_REFERENCE_160: which C# box feeds PixelInBoundingBox */
  float screen_w, screen_h;    /* Screen.width/height used by ParseBoxes / DrawBoxes */
  int32_t image_w, image_h;    /* imageWidth/imageHeight argument of DrawMask / DrawSingleMask */
  int32_t first, count;        /* detection range over the compacted batch; count <= 0 -> all */
  float threshold;             /* mask-probability threshold (IEM:104 _confidenceThreshold): 0 -> the runner's
                                  mask_threshold; negative -> exactly 0 */
} xrseg_mask_params;

/* ---- lifecycle ------------------------------------------------------------------------------ */
/* ↔ ModelLoader.Load + new Worker(model, backend) + warm-up Schedule (IEE:380-387). */
int xrseg_create(const xrseg_config* cfg, xrseg_runner** out);
/* ↔ Worker.Dispose (IEE:303). */
void xrseg_destroy(xrseg_runner* r);
const char* xrseg_last_error(const xrseg_runner* r);   /* r may be NULL: error of the last failed create */
int xrseg_abi_version(void);

/* ---- per-frame path ------------------------------------------------------------------------- */
/* ↔ TextureConverter.ToTensor(tex,640,640,3) + Worker.ScheduleIterable(input) (IEE:370-371).
 * `frames` is HOST memory: batch images of h x w pixels, `stride_bytes` per row, image i at
 * frames + i*h*stride_bytes.  `fmt` = xrseg_pixel_format, optionally | XRSEG_FMT_BOTTOM_UP (row-order contract above:
 * without the flag memory row 0 is the top of the picture).  Asynchronous: returns after enqueueing copy + preprocess +
 * forward + post. */
int xrseg_schedule(xrseg_runner* r, const uint8_t* frames, int w, int h, int stride_bytes, int fmt, int batch);
/* Same with frames already resident in device memory (no host->device copy). */
int xrseg_schedule_device(xrseg_runner* r, const uint8_t* d_frames, int w, int h, int stride_bytes, int fmt, int batch);
/* ↔ the MoveNext loop + IsReadbackRequestDone polling (IEE:397,434-442): 0 running, 1 done, <0 error. */
int xrseg_poll(xrseg_runner* r);
/* Blocks until the scheduled run is complete; returns 1 or <0. */
int xrseg_wait(xrseg_runner* r);
/* Per-frame detection counts of the finished run (n ints, n = scheduled batch). */
int xrseg_counts(xrseg_runner* r, int32_t* counts, int cap);
/* Capacity flags of the finished run: bit 0 = a frame had more score-filtered candidates than max_candidates,
 * bit 1 = a frame kept more boxes than max_det (0 = the results are exactly the unlimited NMS of the reference). */
int xrseg_overflow(xrseg_runner* r);
/* ↔ Worker.PeekOutput(i) (IEE:426): idx 0 boxes f32 [N,4] cx,cy,w,h; 1 labels i32 [N]; 2 coefs f32 [N,32];
 * 3 mask probabilities f32 [N,160,160].  Rows in NMS (descending score) order per frame. */
int xrseg_peek_output(xrseg_runner* r, int idx, xrseg_tensor_view* view);
/* ↔ Tensor.ReadbackRequest + ReadbackAndClone (IEE:427,446-449): blocking copy into caller memory. */
int xrseg_readback(xrseg_runner* r, int idx, void* dst, size_t cap_bytes, int64_t* shape, int* rank);
/* ↔ IEExecutor.ParseBoxes (IEE:529-559) / IEBoxer.DrawBoxes (IEB:37-81).  Per frame the C# caps apply. */
int xrseg_decode(xrseg_runner* r, float screen_w, float screen_h, int convention, xrseg_box* out, int cap, int* n);
/* ↔ IEMasker.DrawMask / DrawSingleMask + PixelInBoundingBox (IEM:82-119,124-196,232-247).  Returns the number of masks
 * written.  out == NULL: the masks are computed into the runner's device scratch only (no device->host copy). */
int xrseg_masks(xrseg_runner* r, const xrseg_mask_params* p, uint8_t* out, size_t cap_bytes);
/* Extension: what a frame loop reads back, in ONE call and ONE synchronisation -- waits for the run like xrseg_wait, then
 * output_0 (boxes f32 [N,4]) -> boxes, output_1 (labels i32 [N]) -> labels and, when p and masks are given, the masks of
 * xrseg_masks(p) -> masks.  Replaces ReadbackRequest x N + the IsReadbackRequestDone polling loop of IEE:419-456 for callers that
 * do not need the four raw tensors.  Any of boxes / labels / masks may be NULL.  Returns N (the number of detections over the
 * batch; counts per frame: xrseg_counts) or a negative error (XRSEG_ERR_CAPACITY: cap_dets < N or masks_cap too small). */
int xrseg_collect(xrseg_runner* r, float* boxes, int32_t* labels, int cap_dets, const xrseg_mask_params* p, uint8_t* masks,
                  size_t masks_cap);
/* Kept anchor indices (0..8399) and scores of the finished run, compacted like output_0. */
int xrseg_keep_indices(xrseg_runner* r, int32_t* idx, float* scores, int cap);

/* ---- the step after the path (SURVEY.md §8f N3) ------------------------------------------------ */
/* ↔ the fields IEExecutor hands to DepthExtractionJob (IEE:623-644): depth texture geometry, sampling step (_samplingStep,
 * XRScene.unity:1259 = 5), _maxPoints (8000), _confidenceThreshold, Screen size, the depth camera pose and intrinsics. */
typedef struct xrseg_depth_params {
  uint32_t struct_size;
  int32_t detection;           /* row of the compacted outputs (targetIndex of ExtractDepthData, IEE:561) */
  int32_t depth_w, depth_h;    /* depth texture size; texels are IEEE half floats in metres */
  int32_t sampling_step;       /* 0 -> 5 */
  int32_t max_points;          /* 0 -> 8000 */
  float confidence_threshold;  /* 0 -> the runner's mask threshold (0.5) */
  float screen_w, screen_h;
  float camera_position[3];    /* _depthCameraPose */
  float camera_rotation[4];    /* _depthCameraRot as x, y, z, w */
  float focal_length[2], principal_point[2], sensor_resolution[2];
} xrseg_depth_params;
/* ↔ ExtractDepthData + DepthExtractionJob.Execute + CollectJobResults (IEE:561-667): world-space points of the target's
 * mask.  depth_host: depth_w*depth_h half floats (host memory); out_xyzd: [cap][4] floats (x, y, z, depth in metres) in
 * sample order, at most max_points.  The 160x160 mask is read on the device (output_3), never copied to the host. */
int xrseg_extract_points(xrseg_runner* r, const xrseg_depth_params* p, const uint16_t* depth_host, float* out_xyzd, int cap,
                         int* n);
/* ↔ the locked-target re-association of ProcessInferenceResult (IEE:488-507): among the first 50 boxes (ParseBoxes) of
 * `frame`, the nearest one whose label equals locked_label; *best_index = -1 when none is closer than max_dist (300). */
int xrseg_associate(xrseg_runner* r, int frame, float locked_center_x, float locked_center_y, int locked_label, float screen_w,
                    float screen_h, float max_dist, int* best_index, float* best_dist);

/* ---- host helpers ------------------------------------------------------------------------------ */
/* Page-locked host memory for frame / result buffers (cudaHostAlloc); NULL on failure. */
void* xrseg_host_alloc(size_t bytes);
void xrseg_host_free(void* p);
/* Number of usable sm_100 devices (0 when there is no GPU: nothing in this library can run then). */
int xrseg_device_count(void);

/* ---- model introspection (host side builds weight packs from this) ---------------------------- */
typedef struct xrseg_layer_info {
  char name[32];
  int32_t cin, cout, k, stride, groups, act, transposed, h_in, w_in;
} xrseg_layer_info;
int xrseg_layer_count(int model_scale);
int xrseg_layer_info_get(int model_scale, int index, xrseg_layer_info* info);
/* The same for a model trained on num_classes classes (1..1024): the class branch is max(ch[2], min(num_classes, 100))
 * wide and the three *.cls.2 convolutions have num_classes outputs; names and order do not change.  The two functions
 * above are the num_classes = 80 case. */
int xrseg_layer_count_nc(int model_scale, int num_classes);
int xrseg_layer_info_get_nc(int model_scale, int num_classes, int index, xrseg_layer_info* info);
/* Scale ('n' / 's', from the width of the first convolution) and class count (from the three *.cls.2 convolutions, which
 * must agree and lie in 1..1024) of a weight pack or .sentis asset; host only.  XRSEG_ERR_WEIGHTS otherwise. */
int xrseg_weights_info(const void* data, size_t bytes, int32_t* model_scale, int32_t* num_classes);
/* Class count of a runner's model. */
int xrseg_num_classes(const xrseg_runner* r);

/* ---- .sentis asset introspection (↔ ModelLoader.Load, IEE:382; host only, no GPU needed) --------- */
/* Number of biased convolutions in the asset and the thresholds baked into its NonMaxSuppression layer
 * (IEModelEditorConverter.cs:76); 0 thresholds when the graph has no NMS. */
int xrseg_sentis_info(const void* data, size_t bytes, int32_t* n_convs, float* iou_threshold, float* score_threshold);
/* Dequantized ((q - zp) * scale, like the graph's DequantizeUint8 layers) weights / bias of convolution `index` in chain
 * order.  w_shape4: [cout,cin/g,kh,kw] ([cin,cout,kh,kw] when transposed).  Returns the weight element count. */
int xrseg_sentis_layer(const void* data, size_t bytes, int index, float* w, size_t w_cap, float* b, size_t b_cap,
                       int32_t* w_shape4, int32_t* transposed);

/* ---- timing ---------------------------------------------------------------------------------- */
/* Device time (ms, CUDA events on the runner's stream) of the last finished run: [0] whole run,
 * [1] preprocess, [2] network, [3] decode+NMS, [4] masks. */
int xrseg_last_timings(xrseg_runner* r, float* ms, int n);
/* Number of kernel launches (graph nodes) one scheduled run issues. */
int xrseg_launch_count(xrseg_runner* r);
/* CUDA events on the runner's own stream (slot 0..7): record now / milliseconds between two recorded slots.
 * Lets a harness time a sequence of xrseg_schedule* calls on the device, on the stream the kernels run on. */
int xrseg_event_record(xrseg_runner* r, int slot);
int xrseg_event_elapsed_ms(xrseg_runner* r, int slot_a, int slot_b, float* ms);
/* Blocks until everything enqueued on the runner's stream has finished. */
int xrseg_sync(xrseg_runner* r);
/* Per-kernel device time of the network + post-processing of the last scheduled input (frames must still be
 * resident): replays each launch `iters` times between CUDA events.  ms[i] = average ms of launch i, names[i*32]
 * its label, flops[i] / bytes[i] its algorithmic work.  Returns the number of launches. */
int xrseg_profile_ops(xrseg_runner* r, int iters, float* ms, char* names, double* flops, double* bytes, int cap);

/* The parity / probe hooks used by tests/ and tools/ (xrseg_debug_*) are NOT part of this library: they are declared in
 * xrseg_debug.h and exported only by libxrseg_debug.so, a second build of the same sources with -DXRSEG_DEBUG_API. */

#ifdef __cplusplus
}
#endif
#endif /* XRSEG_H_ */
