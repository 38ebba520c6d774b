/*
 * rf_b200.h -- C ABI of librf_b200.so: the B200-native (sm_100a) RetinaFace mnet25 detect path.
 *
 * This is the drop-in boundary.  The reference has no FFI layer of its own: its seam is the
 * C++ class `TrtRetinaFaceNet` plus three free CUDA launchers used by `RetinaFace`
 * (retinaface/RetinaFace.cpp:4-6,275-291,584-608,655,670-684).  Each entry point below names
 * the reference interface it replaces.  Plain pointers and sizes only; no C++/torch types.
 *
 * Conventions
 *   - every function returns RF_OK (0) or a negative rf_status; rf_last_error() gives text.
 *     Nothing aborts/exits (the reference abort()s/exit()s/throws: trtutility.h:9-16,
 *     trtnetbase.cpp:201-204, RetinaFace.cpp:327-335).
 *   - one handle = one device + one stream; calls on a handle are serialised by the caller
 *     (the reference is single-threaded and non re-entrant, SURVEY.md 8b).
 *   - there is NO CPU fallback: every compute entry point runs CUDA kernels on the handle's
 *     device and fails with RF_ERR_CUDA if that is impossible.
 *   - images are u8 BGR HWC like cv::Mat (RetinaFace.cpp:594), results are FaceDetectInfo
 *     records (RetinaFace.h:37-42) in network-input pixel coordinates (RetinaFace.cpp:707).
 */
#ifndef RF_B200_H
#define RF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RF_B200_ABI_VERSION 2     /* 2: rf_config gained prototxt_path / cache_path / network (appended) */

typedef enum rf_status {
    RF_OK = 0,
    RF_ERR_INVALID_ARG = -1,
    RF_ERR_IO = -2,          /* model file missing / unreadable */
    RF_ERR_MODEL = -3,       /* caffemodel does not hold the mnet25 topology */
    RF_ERR_CUDA = -4,        /* CUDA runtime / launch failure (text in rf_last_error) */
    RF_ERR_NO_DEVICE = -5,   /* no sm_100 device: the library has no CPU path */
    RF_ERR_CAPACITY = -6,    /* batch / image larger than the handle was created for */
    RF_ERR_UNSUPPORTED = -7
} rf_status;

/* Arithmetic of the network body.  Head 1x1 convs, softmax, decode and NMS are always FP32. */
typedef enum rf_precision {
    RF_PREC_FP32 = 0,   /* FP32 storage + FP32 SIMT math: the tight-parity mode */
    RF_PREC_FP16 = 1,   /* FP16 NHWC activations/weights, FP32 accumulate (tcgen05 where GEMM-shaped) */
    RF_PREC_INT8 = 2    /* INT8 activations with the TensorRT calibration-table scales */
} rf_precision;

/* == FaceDetectInfo (RetinaFace.h:37-42): score, rect(x1,y1,x2,y2), pts.x[5], pts.y[5]. */
typedef struct rf_face {
    float score;
    float x1, y1, x2, y2;
    float lx[5];
    float ly[5];
} rf_face;

/* Device/all-gather record: rf_face + the anchor's emission index (stride 32->16->8, anchor,
 * row-major position: the order of the reference's decode loop, RetinaFace.cpp:666-690).
 * 64 bytes. */
typedef struct rf_det {
    rf_face face;
    int32_t anchor_index;
} rf_det;

typedef struct rf_config {
    const char *caffemodel_path;   /* replaces buildTrtContext(prototxt, caffemodel), RetinaFace.cpp:276 */
    const char *int8_table_path;   /* TensorRT EntropyCalibration2 cache (trtnetbase.cpp:13) or NULL */
    int precision;                 /* rf_precision */
    int net_w, net_h;              /* network input size (prototxt line 7 in the reference); multiples of 32 */
    int max_batch;                 /* reference: maxBatchSize = 8 (trtretinafacenet.cpp:21) */
    int max_faces;                 /* per-image output capacity (faces kept after NMS); 0 -> 256 */
    int device;                    /* CUDA device ordinal */
    int max_image_w, max_image_h;  /* largest caller image (reference: 4096x3072, RetinaFace.cpp:325); 0 -> net size */
    unsigned flags;                /* RF_FLAG_* */
    int streams;                   /* execution contexts the asynchronous entry points rotate through so that
                                      consecutive batches overlap on the GPU; 0 -> RF_MAX_STREAMS (8).  The blocking
                                      rf_detect_batch always uses context 0.  1 selects the latency-oriented layer plan. */
    const char *prototxt_path;     /* optional: the Caffe prototxt of the model (buildTrtContext's first argument, RetinaFace.cpp:276).
                                      Parsed as protobuf text, checked to be the RetinaFace mnet25 graph, and its per-layer
                                      parameters (kernel, stride, group, bias_term, BatchNorm eps, ReLU) drive the weight folding;
                                      net_w / net_h == 0 take the input size from it (trtnetbase.cpp:163-187).  NULL: built-in graph. */
    const char *cache_path;        /* optional: file caching the folded model (the reference's engine cache, trtnetbase.cpp:205-243,
                                      which is never invalidated); reused only for the exact caffemodel (+ prototxt) bytes it was
                                      made from, rewritten otherwise.  NULL: no cache. */
    const char *network;           /* optional: the reference's network name (RetinaFace.cpp:205: "net3" default).  Names whose
                                      configuration the reference itself cannot run (net5, net6 ...: :266-268) or that need more
                                      anchors than the shipped models have (net3a) are refused with RF_ERR_UNSUPPORTED. */
} rf_config;

#define RF_FLAG_NO_GRAPH      0x1u  /* launch kernels directly instead of replaying a CUDA graph */
#define RF_FLAG_NO_TENSORCORE 0x2u  /* FP16: use the SIMT kernels for GEMM-shaped layers too (implies RF_FLAG_SIMT_STEM) */
#define RF_FLAG_SIMT_STEM     0x4u  /* FP16 / INT8: run all three layers of the stem on CUDA cores (FP32 conv0 weights) */
#define RF_FLAG_DW_1D         0x8u  /* FP16 / INT8: linear (1-D) tiles for every depthwise+pointwise layer, also on large maps */
#define RF_FLAG_NPP_RESIZE    0x20u /* letter-box with the reference's NPP branch semantics (USE_NPP: nppiResizeSqrPixel_8u_C3R,
                                       NPPI_INTER_SUPER, resizeconvertion.cu:279-316) -- coverage-weighted super-sampling, extent
                                       ceil(w f) x ceil(h f) -- instead of its OpenCV branch (cv::resize INTER_LINEAR, RetinaFace.cpp:613) */
#define RF_FLAG_LEGACY_TC     0x10u /* FP16: one round-1 tensor-core kernel per layer (pair) instead of the persistent tile chains
                                       (tile_chain.cuh); the cross-check of the chains */

typedef struct rf_handle_s *rf_handle;

/* Process-wide info, callable without a GPU. */
int rf_abi_version(void);
const char *rf_build_info(void);            /* arch flags etc. */
const char *rf_status_string(int status);

/* Replaces RetinaFace::RetinaFace's engine setup (RetinaFace.cpp:274-302): parses the
 * caffemodel, folds BatchNorm+Scale(+bias) in FP32, repacks weights, allocates device and
 * pinned memory, builds CUDA graphs lazily.  On failure *out = NULL and the message is
 * available from rf_last_error(NULL). */
int rf_create(const rf_config *cfg, rf_handle *out);
void rf_destroy(rf_handle h);
const char *rf_last_error(rf_handle h);     /* h may be NULL: last rf_create error */

/* Library-owned pinned staging for network-sized inputs: max_batch * net_h * net_w * 3 bytes.
 * Writing images here lets rf_detect_batch skip its host-side staging copy. */
uint8_t *rf_pinned_input(rf_handle h);
/* Library-owned DEVICE input buffer of the same shape: a caller that already has its images on
 * the GPU writes them here and passes this pointer to rf_detect_batch_device (no D2D copy). */
uint8_t *rf_device_input(rf_handle h);

/* Replaces RetinaFace::detect / detectBatchImages (RetinaFace.cpp:576-747, 749-940), end to
 * end: host u8 BGR HWC images (any size <= max_image; letter-boxed top-left into the network
 * size, never up-scaled) -> H2D -> network -> decode + threshold + NMS on the GPU -> D2H.
 * `row_strides` in bytes (NULL = packed).  Writes up to max_faces faces per image to
 * out_faces[i * max_faces ...] in descending score order and the count to out_counts[i].
 * out_anchor_index (optional, same layout) receives each face's anchor emission index.
 * Blocking: returns when the results are in the caller's arrays. */
int rf_detect_batch(rf_handle h, const uint8_t *const *bgr_images, const int *widths, const int *heights,
                    const int *row_strides, int n, float score_threshold, float nms_threshold,
                    rf_face *out_faces, int *out_counts, int32_t *out_anchor_index);

/* Pipelined end to end (throughput mode of the same path): rf_submit_batch queues H2D (on a copy
 * stream) + forward + D2H for one batch of NETWORK-SIZED images and returns at once with a ticket;
 * rf_collect_batch blocks until that batch's faces are in the caller's arrays.  Up to
 * RF_PIPELINE_DEPTH batches may be in flight, so the H2D copy of batch i+1 overlaps the kernels of
 * batch i (SURVEY.md 8f-1: host ingest).  Tickets must be collected in submission order.  Source
 * images may be pinned (copied in place) or pageable (staged through the library's pinned ring).
 * Every bgr_images[i] MUST point at net_h * net_w * 3 readable bytes (a packed network-sized image): there are no
 * width / height / stride arguments here -- other sizes go through rf_detect_batch. */
#define RF_MAX_STREAMS 8
#define RF_PIPELINE_DEPTH 6
int rf_submit_batch(rf_handle h, const uint8_t *const *bgr_images, int n, float score_threshold, float nms_threshold,
                    int *ticket);
int rf_collect_batch(rf_handle h, int ticket, rf_face *out_faces, int *out_counts, int32_t *out_anchor_index);

/* Device-resident variant: `dev_bgr` holds n network-sized u8 BGR HWC images (contiguous) in
 * device memory; results stay on the device: *dev_dets -> [max_batch][max_faces] rf_det,
 * *dev_counts -> [max_batch] int32 (kept count, clamped to max_faces).  Asynchronous on the
 * stream of the execution context the call landed on (rf_last_stream; rf_synchronize waits for all).
 * Consecutive calls rotate over the handle's execution contexts, each with its own output buffers: the
 * returned pointers stay valid until `streams` further calls.  This is the buffer a multi-GPU caller
 * all-gathers (SURVEY.md 8e). */
int rf_detect_batch_device(rf_handle h, const uint8_t *dev_bgr, int n, float score_threshold,
                           float nms_threshold, const rf_det **dev_dets, const int32_t **dev_counts);
/* (aligned crops of these results: rf_align_batch_device, below) */

/* f1 ingest, compressed: the reference decodes its test images on the host (cv::imread, main.cpp:18-26) and then copies
 * pixels; here the JPEG bitstreams are decoded ON the GPU (nvJPEG, opened at run time; hardware JPEG engines when the device
 * and the stream allow it, nvJPEG's hybrid back end otherwise) into the same device buffers the pixel path letter-boxes from,
 * so a camera-sized photo crosses PCIe as its compressed bytes.  jpegs[i] / jpeg_bytes[i]: host memory.  Images may have any
 * size up to max_image; out_widths / out_heights (optional) receive the decoded sizes (map-back: RetinaFace.cpp:732-738).
 * Results as rf_detect_batch.  RF_ERR_UNSUPPORTED when libnvjpeg is absent. */
int rf_detect_jpeg_batch(rf_handle h, const uint8_t *const *jpegs, const size_t *jpeg_bytes, int n, float score_threshold,
                         float nms_threshold, rf_face *out_faces, int *out_counts, int32_t *out_anchor_index, int *out_widths,
                         int *out_heights);
/* Decode only (parity / callers that want the pixels): BGR u8, packed rows, into out_bgr (host, out_capacity bytes);
 * out_bgr == NULL just reports the size.  rf_jpeg_backend: "hardware" | "default" | "none" (+ what the last call used). */
int rf_decode_jpeg(rf_handle h, const uint8_t *jpeg, size_t bytes, uint8_t *out_bgr, size_t out_capacity, int *width, int *height);
const char *rf_jpeg_backend(rf_handle h);

/* ---- Multi-GPU (SURVEY.md 8e; the reference is single-GPU: `ctx_id`, RetinaFace.h:89, is never used) --------------------
 * One process (handle) per GPU; the batch is sharded over the ranks, weights are replicated, and the ONLY exchange is an
 * all-gather of the per-image detection records -- fused into the NMS kernel: the CTA that finishes an image stores its kept
 * faces straight into the gather window of every rank (peer device memory over NVLink, mapped with CUDA IPC) and raises a
 * flag there.  Set-up: every rank calls rf_comm_export (allocates its window, fills an opaque 128-byte blob), the caller
 * all-gathers the blobs by any means (MPI, torch.distributed, a file ...), every rank calls rf_comm_init with all of them in
 * rank order.  rf_comm_init_nccl does the blob exchange itself through NCCL (libnccl.so.2 is opened at run time; the id
 * comes from rf_comm_nccl_unique_id on one rank and reaches the others by the caller's means).
 * All ranks must issue the same sequence of *_allgather calls with the same n. */
#define RF_COMM_BLOB_BYTES 128
#define RF_COMM_MAX_WORLD_SIZE 16
int rf_comm_export(rf_handle h, int rank, int world, void *blob);
int rf_comm_init(rf_handle h, const void *blobs /* world x RF_COMM_BLOB_BYTES, rank order */);
int rf_comm_nccl_unique_id(void *out128);
int rf_comm_init_nccl(rf_handle h, const void *nccl_unique_id /* 128 bytes */, int rank, int world);
int rf_comm_info(rf_handle h, int *rank, int *world);
/* rf_detect_batch_device + exchange: asynchronous; *all_dets -> [world][max_batch][max_faces] rf_det and *all_counts ->
 * [world][max_batch] int32 in this rank's gather window (rank r's image i at r * max_batch + i), complete -- every rank's
 * records have landed -- in stream order on rf_last_stream(); valid until 20 further exchanges. */
int rf_detect_batch_device_allgather(rf_handle h, const uint8_t *dev_bgr, int n, float score_threshold, float nms_threshold,
                                     const rf_det **all_dets, const int32_t **all_counts);
/* rf_submit_batch / rf_collect_batch + exchange: out_faces [world * max_batch][max_faces], out_counts [world * max_batch]
 * (host), rank r's image i at r * max_batch + i.  rf_detect_batch_allgather = submit + collect (blocking). */
int rf_submit_batch_allgather(rf_handle h, const uint8_t *const *bgr_images, int n, float score_threshold, float nms_threshold, int *ticket);
int rf_collect_batch_allgather(rf_handle h, int ticket, rf_face *out_faces, int *out_counts, int32_t *out_anchor_index);
int rf_detect_batch_allgather(rf_handle h, const uint8_t *const *bgr_images, int n, float score_threshold, float nms_threshold,
                              rf_face *out_faces, int *out_counts, int32_t *out_anchor_index);

/* Parity/debug: replaces TrtRetinaFaceNet::doInference + blob_by_name (trtretinafacenet.cpp:48-114).
 * Host network-sized images in, the 9 head blobs out in the reference's blob order
 * (trtretinafacenet.cpp:23-31), NCHW float32, each heads_out[k] sized n*C*h*w. */
int rf_forward_heads(rf_handle h, const uint8_t *bgr_net_sized, int n, float *const heads_out[9]);

/* Kernel-level parity: replaces the host decode loop + nms (RetinaFace.cpp:661-726, 439-492)
 * on caller-supplied head blobs (host, layout as rf_forward_heads).  Same outputs as
 * rf_detect_batch plus the pre-NMS candidate count per image (optional). */
int rf_postprocess(rf_handle h, const float *const heads[9], int n, float score_threshold,
                   float nms_threshold, rf_face *out_faces, int *out_counts, int32_t *out_anchor_index,
                   int *out_num_candidates);

/* Test-time augmentation + map-back (SURVEY.md 8f-2; the reference's `scales` parameter, RetinaFace.h:70, is unused and its
 * map-back is commented out, RetinaFace.cpp:730-746).  One image, `nviews` views of it (1..RF_MAX_VIEWS, <= max_batch): view v
 * is the image -- mirrored horizontally when views[v].flip -- letter-boxed into the top-left
 * floor(net_w*shrink) x floor(net_h*shrink) corner of the network input (shrink in (0, 1]; 1 = the plain detect view).
 * All views run as ONE batch; their detections are mapped back to ORIGINAL IMAGE pixels (x * scale_v, mirrored views
 * un-mirrored with left/right landmarks swapped) and merged by one more greedy NMS (same rule and threshold as per view)
 * across views, all on the GPU.  out_faces: [max_faces] in image coordinates; out_view_of (optional, [max_faces]): which view
 * each kept face came from; out_view_scales (optional, [nviews]): the map-back factor of each view.
 * views = {{1.0f, 0}} is detect + map-back. */
typedef struct rf_view {
    float shrink;
    int32_t flip;
} rf_view;
#define RF_MAX_VIEWS 16
int rf_detect_views(rf_handle h, const uint8_t *bgr, int width, int height, int row_stride, const rf_view *views, int nviews,
                    float score_threshold, float nms_threshold, rf_face *out_faces, int *out_count, int32_t *out_view_of,
                    float *out_view_scales);

/* Landmark-aligned face crops: insightface's norm_crop -- a similarity transform fitted (least squares, no reflection, FP64)
 * from a face's five landmarks to a template, then cv2.warpAffine(img, M, (crop_w, crop_h), INTER_LINEAR, BORDER_CONSTANT, 0)
 * -- on the GPU, byte for byte what OpenCV computes with the same M.  The crop is what a recognizer (ArcFace and its relatives)
 * takes.  One kernel launch per call aligns the first min(count, max_crops) faces of every image, in score order, straight
 * from the full-resolution source images the detector read; it is not part of the forward graph. */
#define RF_CROP_U8_BGR  0   /* [crop_h][crop_w][3] u8 BGR: norm_crop's output */
#define RF_CROP_F16_RGB 1   /* [3][crop_h][crop_w] FP16 of (v - mean) * scale, RGB planes: a recognizer's input tensor */
typedef struct rf_align_spec {
    int crop_w, crop_h;         /* 1..1024; with the default template both must be multiples of 112 */
    float dst_x[5], dst_y[5];   /* landmark template in crop pixels; all zero -> the ArcFace 112 template scaled by crop / 112
                                   (insightface estimate_norm) */
    int max_crops;              /* per image, 1..max_faces: crops of the top-scoring faces */
    int layout;                 /* RF_CROP_* */
    float mean, scale;          /* RF_CROP_F16_RGB only (insightface: 127.5, 1/127.5) */
} rf_align_spec;

/* rf_detect_batch + aligned crops of the first min(out_counts[i], max_crops) faces of each image, sampled from the caller's
 * ORIGINAL image (any size <= max_image; at most raw_slots -- max_batch, capped at 2 GiB of image buffers -- of them not
 * network-sized, RF_ERR_CAPACITY otherwise).  Faces / counts / anchor indices exactly as rf_detect_batch (network-input
 * pixels); out_scales (optional) [n]: the map-back factor to image pixels; out_crops (host) [n][max_crops][crop] in the spec's
 * layout; out_affine (optional) [n][max_crops][6] doubles, the image -> crop matrix of each crop.  Slots past the count are not
 * written.  Blocking. */
int rf_detect_align_batch(rf_handle h, const uint8_t *const *bgr_images, const int *widths, const int *heights,
                          const int *row_strides, int n, float score_threshold, float nms_threshold, const rf_align_spec *spec,
                          rf_face *out_faces, int *out_counts, int32_t *out_anchor_index, float *out_scales,
                          void *out_crops, double *out_affine);
/* Device-resident: after rf_detect_batch_device(h, dev_bgr, n, ...) align from the same network-sized device images and the
 * records it returned (dev_dets [n][max_faces], dev_counts [n]).  Enqueued on rf_last_stream(); dev_crops / dev_affine
 * (optional) are caller-owned device memory laid out as above; slots past the count are not written. */
int rf_align_batch_device(rf_handle h, const uint8_t *dev_bgr, int n, const rf_det *dev_dets, const int32_t *dev_counts,
                          const rf_align_spec *spec, void *dev_crops, double *dev_affine);

/* Preprocess parity: replaces imageROIResize8U3C + the OpenCV branch (RetinaFace.cpp:593-647):
 * letter-boxes one host image into a host net_h*net_w*3 u8 BGR buffer using the GPU kernel. */
int rf_preprocess(rf_handle h, const uint8_t *bgr, int width, int height, int row_stride, uint8_t *out_net_sized);

/* Introspection. */
int rf_get_net_size(rf_handle h, int *net_w, int *net_h, int *max_batch, int *max_faces);
int rf_num_anchors(rf_handle h);            /* per image: 8,232 @448x448, 47,040 @1280x896 */
void *rf_stream(rf_handle h);               /* cudaStream_t */
int rf_synchronize(rf_handle h);            /* all execution contexts */
/* rf_stream() is context 0's stream.  rf_fence() orders it after everything queued so far on every context
 * (for CUDA-event timing of a run of rf_detect_batch_device calls); rf_last_stream() is the stream the last
 * rf_detect_batch_device call was issued on (to order a collective on that call's device outputs). */
int rf_fence(rf_handle h);
void *rf_last_stream(rf_handle h);
/* Number of kernel launches (graph kernel nodes) one rf_detect_batch_device of batch n issues. */
int rf_launches_per_batch(rf_handle h, int n);
/* Names + device times (ms, CUDA events, direct launches) of each kernel of one forward of
 * batch n: fills up to cap entries, returns the count.  For bench.py's roofline line. */
int rf_profile_layers(rf_handle h, int n, int iters, char (*names)[64], float *ms, double *bytes, double *flops, int cap);

/* INT8 entropy calibration -- replaces the reference's offline INT8-Calibration-Tool (calibrationtable.cpp:399-583):
 * runs the n network-sized u8 BGR host images through an RF_PREC_FP32 handle twice (absmax, then 2048-bin histograms of
 * every activation tensor), searches the KL-optimal clipping threshold per tensor and writes a table in the reference's
 * own TensorRT cache format ("TRT-5102-EntropyCalibration2", one "<caffe top>: <hex float32 scale>" line per tensor) that
 * rf_create(RF_PREC_INT8) -- or the reference's Int8EntropyCalibrator2 reader (trtnetbase.cpp:31-44) -- consumes. */
int rf_calibrate_int8(rf_handle h, const uint8_t *bgr_net_sized, int n_images, const char *out_table_path);
/* Host-only: the threshold search of the calibrator on one histogram (returns the threshold in bins). */
double rf_kl_threshold_bins(const unsigned *hist, int bins, int levels);

/* Host-only (works without a GPU): the layer plan rf_create would build for `cfg`, one text line per kernel launch of a
 * forward plus the geometry / shared-memory budget of every persistent tile chain.  Returns the launch count. */
int rf_plan_describe(const rf_config *cfg, char *out, int cap);

/* Debug / parity aids (not part of the drop-in surface): fetch a materialised activation by its
 * Caffe top name (e.g. "mobilenet0_relu10_fwd", "_plus0", "rf_c1_det_concat_relu") as NCHW
 * float32 after a forward; rf_debug_keep_all disables activation-buffer reuse so every tensor
 * of the last forward survives. */
int rf_debug_get_tensor(rf_handle h, const char *name, int n, float *out_nchw, int *c, int *hh, int *ww);
int rf_debug_keep_all(rf_handle h);
/* Host-only (works without a GPU): the folded FP32 weights / bias of one convolution layer as the
 * engine holds them; dims = {cout, cin/groups, k, k}.  For CPU-side tests of the model front end. */
int rf_model_inspect(const char *caffemodel_path, const char *layer, float *w, int wcap, float *b, int bcap, int dims[4]);
/* Host-only model front end (SURVEY.md 8f-4).  rf_model_load: the complete load path of rf_create -- cache lookup, prototxt parse +
 * graph check, file-driven folding, cache write -- without a device; *cache_status: 0 no cache, 1 miss (written), 2 hit,
 * 3 stale (rewritten); input_dims: N, C, H, W of the prototxt (zeros without one); then rf_model_inspect semantics for `layer`
 * (may be NULL).  rf_network_config: the reference's network-name switch (RetinaFace.cpp:211-268): FPN strides, anchor scales per
 * level (2 each), ratios; RF_ERR_UNSUPPORTED where the reference prints "please reconfig anchor_cfg". */
int rf_model_load(const char *caffemodel_path, const char *prototxt_path, const char *cache_path, int *cache_status, int input_dims[4],
                  const char *layer, float *w, int wcap, float *b, int bcap, int dims[4]);
int rf_network_config(const char *network, int *num_levels, int strides[3], int scales[6], float ratios[2], int *num_ratios);
/* Cache state of a handle's model load (the enum above). */
int rf_cache_status(rf_handle h);

#ifdef __cplusplus
}
#endif
#endif /* RF_B200_H */
