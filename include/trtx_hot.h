/*
 * trtx_hot.h -- C ABI of the B200-native detection hot path (libtrtx_hot.so).
 *
 * This is the drop-in boundary: every entry point below is what a TensorRT plugin's
 * enqueue()/getWorkspaceSize() (or the driver's cuda_* helper) in wang-xinyu/tensorrtx
 * binds to.  Plain pointers and sizes only; all pointers named *_dev are DEVICE pointers
 * owned by the caller (TensorRT owns inputs/outputs/workspace, SURVEY.md section 8b);
 * nothing is allocated, freed, retained or synchronised inside an enqueue; every call is
 * re-entrant and ordered on the given stream.  Return value: 0 = success (the reference's
 * enqueue() convention, yolov8/plugin/yololayer.cu:171), non-zero = TRTX_ERR_*; the library
 * never throws and never asserts.
 *
 * Reference citations are relative to /root/reference (wang-xinyu/tensorrtx @ 3ff22bb4).
 * The header-only TensorRT adapters that forward the IPluginV2DynamicExt / IPluginV2IOExt /
 * IPluginV2Ext virtuals to these functions live in include/trtx_plugins.h; the binding a
 * maintainer adds on the reference side is shown in INTEGRATION.md.
 */
#ifndef TRTX_HOT_H
#define TRTX_HOT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define TRTX_API __declspec(dllexport)
#else
#define TRTX_API __attribute__((visibility("default")))
#endif

/* cudaStream_t, spelled without <cuda_runtime.h> so that C / cgo / ctypes callers can include this. */
typedef void* trtx_stream_t;

enum {
    TRTX_OK = 0,
    TRTX_ERR_INVALID = 1,     /* malformed params / null pointer */
    TRTX_ERR_WORKSPACE = 2,   /* workspace too small (the reference throws here, rcnn/cuda_utils.h:22-24) */
    TRTX_ERR_CUDA = 3,        /* a launch failed; see trtx_last_cuda_error() */
    TRTX_ERR_UNSUPPORTED = 4, /* parameter combination outside what the kernels cover */
};

#define TRTX_MAX_LEVELS 8

TRTX_API const char* trtx_version(void);
/* cudaError_t of the last failing launch on this thread (0 if none). */
TRTX_API int trtx_last_cuda_error(void);
/* sizeof() of the parameter structs as THIS library was compiled, so that an FFI binding (ctypes, cgo, ...) can check its
 * mirror of the layout: which = 0 trtx_yolo_params, 1 trtx_nms_params, 2 trtx_retina_params, 3 trtx_image_desc,
 * 4 trtx_mask_params; anything else 0. */
TRTX_API size_t trtx_abi_sizeof(int which);

/* =====================================================================================
 * 1. YoloLayer_TRT  -- fused per-anchor sigmoid / argmax / gate / box decode / compaction
 *    replaces CalDetection + forwardGpu of
 *      yolov8/plugin/yololayer.cu:178-316 (anchor-free: yolov8, yolo11, yolov12, yolov13, yolov9/10 subsets)
 *      yolov5/plugin/yololayer.cu:161-227 (anchor-based: yolov5, yolov7, yolov5-lite, yolop)
 * ===================================================================================== */
enum {
    TRTX_YOLO_V8 = 0,
    TRTX_YOLO_V5 = 1,
    /* SURVEY 8f rank 4 -- older / other YoloLayer variants through the same scan / pack / NMS kernels: */
    TRTX_YOLO_V3 = 2,  /* yolov3, yolov3-spp, yolov4 (yolov3-spp/yololayer.cu:148-191): anchor-based like V5, but box =
                          ((col + sigmoid(x)) * stride, ..., exp(w) * anchor_w, ...), class AND objectness gated, rows of 7
                          floats x,y,w,h, det_confidence, class_id, class_confidence (yololayer.h:47-53).  `strides` and
                          `anchors` are both used; det_floats >= 7 */
    TRTX_YOLO_V26 = 3, /* yolo26 NMS-free gatherKernel (yolo26/plugin/yololayer.cu:178-245): ONE input
                          [batch, anchors, 4 + num_classes (+1 angle when is_obb)], row-major per anchor, scores are
                          probabilities already; argmax `>` from (0, class -1), rows with score < gate dropped, 90-float
                          rows, everything the kernel does not write is zero (the reference memsets the buffer).
                          num_levels = 1, grid_h[0] * grid_w[0] = anchor count.  The reference decodes image 0 only
                          (":185 TODO"); this build decodes every image of the batch */
};
enum { TRTX_F32 = 0, TRTX_F16 = 1 };

typedef struct trtx_yolo_params {
    int32_t variant;     /* TRTX_YOLO_V8 | TRTX_YOLO_V5 | TRTX_YOLO_V3 | TRTX_YOLO_V26 */
    int32_t num_classes; /* combinedInfo[0] (yolov8/src/block.cpp:268) | netinfo[0] (yolov5/src/model.cpp:249) */
    int32_t net_w;       /* kInputW */
    int32_t net_h;       /* kInputH */
    int32_t max_out;     /* kMaxNumOutputBbox: capacity of the plugin output, rows per image */
    int32_t det_floats;  /* sizeof(Detection)/4 of the model dir: 90 (yolov8/include/types.h:4-12),
                            38 (yolov5/src/types.h:11-16), 6 (yolov7/10/13: yolov7/include/types.h:11-16),
                            7 (yolov3-spp/yololayer.h:47-53) */
    int32_t num_levels;  /* number of input tensors (strides) */
    int32_t grid_h[TRTX_MAX_LEVELS]; /* v8: net_h/stride (yololayer.cu:294); v5: YoloKernel.height */
    int32_t grid_w[TRTX_MAX_LEVELS];
    int32_t strides[TRTX_MAX_LEVELS];   /* v8 only (combinedInfo[9..]) */
    float anchors[TRTX_MAX_LEVELS][6];  /* v5 only: YoloKernel.anchors (yolov5/src/types.h:5-9) */
    int32_t is_seg;      /* copy 32 mask coefficients */
    int32_t is_pose;     /* v8: decode num_kpts keypoints */
    int32_t is_obb;      /* v8: rotated box */
    int32_t num_kpts;    /* combinedInfo[1] */
    float kpt_thresh;    /* combinedInfo[2] (int-truncated by the reference builder, block.cpp:271) */
    float gate;          /* 0.1f: literal of yolov8 yololayer.cu:203 / kIgnoreThresh yolov5 config.h:38 / IGNORE_THRESH
                            yolov3-spp yololayer.h:15; V26: the confidence threshold (d_confThreshold, yololayer.cu:9,32) */
    int32_t in_dtype;    /* TRTX_F32 (parity mode, what the reference accepts, yololayer.h:32-35) | TRTX_F16 */
    /* Launch tuning of the scan kernel.  Plain per-call data: the library keeps NO mutable state, so concurrent enqueues
     * (TensorRT calls enqueue() on clones from several threads, SURVEY 8b "Threading") with different tunings are
     * independent.  0 everywhere -- what memset / trtx_yolo_params_init_v8 leave -- selects the defaults taken from the
     * B200 sweep in profiles/.  A combination that is not built returns TRTX_ERR_UNSUPPORTED. */
    int32_t tune_class_slices;   /* warps of a CTA splitting the class range: 1, 2, 4, 8; 0 = 2 */
    int32_t tune_rows_in_flight; /* channel rows loaded per group; 0 = 5 (fp16 inputs, 8 anchors per lane: 10).  Built (slices, rows): (1,8) (1,16) (2,4) (2,5)
                                    (2,8) (2,10) (2,20) (4,4) (4,5) (4,10) (4,20) (8,5) (8,10) */
    int32_t tune_tma_pipeline;   /* 1: persistent TMA-fed scan (v8 layout, 16-byte aligned levels); 0 = register scan */
    int32_t tune_tma_stages;     /* cap on its pipeline stages; 0 = as many as fit (15) */
    int32_t tune_box_prefetch;   /* box rows of a tile: 1 on demand, 2 L2 prefetch, 3 into registers up front; 0 = 2 */
    int32_t tune_nms_threads;    /* threads per NMS CTA of the fused / split decode + NMS calls: 1024 (every case) or 512
                                    (half an SM: greedy mode, axis-aligned boxes, max_out <= 1024, no gather fused into
                                    the NMS); 0 = 1024.  Both give identical outputs. */
} trtx_yolo_params;

/* Fill grid_h/grid_w from net size and strides (v8) -- convenience, mirrors yololayer.cu:292-296. */
TRTX_API int trtx_yolo_params_init_v8(trtx_yolo_params* p, int num_classes, int net_w, int net_h, int max_out,
                                      const int* strides, int num_levels);

/* Scratch bytes for trtx_yolo_decode_enqueue / trtx_yolo_decode_nms_enqueue at `batch` images.
 * (The reference plugin needs none, yololayer.h:22; this build stages candidates per tile so that
 *  compaction is atomic-free and deterministic.) */
TRTX_API size_t trtx_yolo_workspace_size(const trtx_yolo_params* p, int batch);

/* Drop-in for YoloLayerPlugin::enqueue (yolov8/plugin/yololayer.cu:167-172, yolov5 :229-232).
 *  inputs_dev[l] : level-l tensor [batch, C_l, grid_h*grid_w], channel-major, fp32 (or fp16)
 *  output_dev    : [batch, 1 + max_out*det_floats] fp32: count, Detection rows.
 * Rows appear in ascending anchor order (deterministic; the reference's order is atomicAdd arrival).
 * count is clamped to max_out (the reference lets it run past, which overruns host readers). */
TRTX_API int trtx_yolo_decode_enqueue(const trtx_yolo_params* p, int batch, const void* const* inputs_dev,
                                      float* output_dev, void* workspace_dev, size_t workspace_bytes,
                                      trtx_stream_t stream);

/* =====================================================================================
 * 2. NMS -- sort + greedy class-aware NMS, one CTA per image, all images in one launch.
 *    replaces the host nms()/batch_nms() of yolov8/src/postprocess.cpp:94-129,
 *    yolov5/src/postprocess.cpp:49-80, retinaface/common.hpp:110-130 and the device
 *    cuda_decode()+cuda_nms() of yolov8/src/postprocess.cu:168-179 (batch 1 only there).
 * ===================================================================================== */
enum {
    TRTX_BOX_LTRB = 0,   /* yolov8 Detection: x1,y1,x2,y2; IoU of postprocess.cpp:71-85 */
    TRTX_BOX_CXCYWH = 1, /* yolov5 Detection: cx,cy,w,h;   IoU of yolov5 postprocess.cpp:30-43 */
    TRTX_BOX_RETINA = 2, /* retinaface: x1,y1,x2,y2, +1e-6f in the denominator, single class (common.hpp:91-104) */
    TRTX_BOX_OBB = 3,    /* yolov8-obb Detection: cx,cy,w,h + angle = the FIRST extra float (extra_floats >= 1,
                            extra_offset = 89 for plugin rows); greedy = nms_obb / probiou `>=`
                            (postprocess.cpp:303-385), one-shot = nms_kernel_obb / box_probiou `>`
                            (postprocess.cu:113-166).  Plugin-row source only (not the fused tile source). */
};
enum {
    TRTX_NMS_GREEDY = 0,  /* CPU nms() semantics (the contract, SURVEY.md section 7 "Hard parts") */
    TRTX_NMS_ONESHOT = 1, /* nms_kernel semantics, yolov8/src/postprocess.cu:89-111 */
};

#define TRTX_NMS_MAX_ROWS 2048 /* rows per image the NMS kernel sorts on chip */

typedef struct trtx_nms_params {
    int32_t box_format;  /* TRTX_BOX_* */
    int32_t mode;        /* TRTX_NMS_* */
    float conf_thresh;   /* rows with !(conf > conf_thresh) are dropped (kConfThresh 0.5 / retinaface 0.1 rounded
                            so that the float compare equals the reference's double compare) */
    float nms_thresh;    /* kNmsThresh 0.45 / 0.4 */
    int32_t max_det;     /* K: rows of the compact output per image (kMaxNumOutputBbox) */
    int32_t class_aware; /* 1: only same-class rows interact (yolo); 0: single class (retinaface) */
    int32_t tie_break_x0; /* 1: equal conf ordered by box[0] ascending (yolov8 cmp, postprocess.cpp:87-92); 0: none */
    int32_t extra_floats; /* floats copied verbatim from each source row into the output row after `keep`
                             (retinaface: 10 landmarks; yolo seg: 32 mask coefficients); 0 for plain det */
    int32_t extra_offset; /* offset (floats) of the first extra in the source row (retinaface 5, yolo seg 6) */
} trtx_nms_params;

/* Compact detection output: [batch, 1 + max_det*R] fp32, R = 7 + extra_floats:
 * count, (x0,x1,x2,x3,conf,cls,keep, extras...)*   (R = 7 is the layout of yolov8/include/types.h:18-19 +
 * postprocess.cu:64-71; box in the input's format).  Rows are ordered class asc then conf desc -- the
 * order of the reference's `res` vector (std::map iteration + std::sort).
 * GREEDY: only kept rows are written (keep=1), count = number kept.  ONESHOT: all rows above
 * conf_thresh, keep flag 0/1, count = rows.  Rows >= count are zero.
 * Rows entering NMS:
 *   trtx_nms_enqueue: every row i < min(count, max_rows) above conf_thresh, exactly like the reference's nms(), as long
 *     as max_rows <= TRTX_NMS_MAX_ROWS; with a larger max_rows (e.g. RetinaFace's 16800 priors) the TRTX_NMS_MAX_ROWS
 *     highest-confidence rows above conf_thresh enter (ties at the cut: lower row index first) -- the reference has no
 *     such cap, so results only differ when more than TRTX_NMS_MAX_ROWS rows of one image pass conf_thresh;
 *   fused / split calls: the first p->max_out candidates in ascending anchor order (= the rows the plugin buffer of
 *     trtx_yolo_decode_enqueue would hold), then the conf_thresh filter: both paths give identical results also when
 *     an image has more than max_out candidates (the reference's choice there is atomicAdd arrival order).
 *     p->max_out <= TRTX_NMS_MAX_ROWS or TRTX_ERR_UNSUPPORTED.
 * keep_index_dev (optional, may be NULL): [batch, max_det] int32 flat anchor id of each written row. */

/* NMS over a plugin-format buffer [batch, 1 + max_rows*det_floats] (drop-in for batch_nms()). */
TRTX_API size_t trtx_nms_workspace_size(const trtx_nms_params* p, int batch, int max_rows);
TRTX_API int trtx_nms_enqueue(const trtx_nms_params* p, int batch, const float* plugin_out_dev, int max_rows,
                              int det_floats, float* compact_out_dev, int32_t* keep_index_dev, void* workspace_dev,
                              size_t workspace_bytes, trtx_stream_t stream);

/* Fused decode + NMS: YoloLayer inputs -> compact detections, no plugin-format round trip. */
TRTX_API int trtx_yolo_decode_nms_enqueue(const trtx_yolo_params* p, const trtx_nms_params* q, int batch,
                                          const void* const* inputs_dev, float* compact_out_dev,
                                          int32_t* keep_index_dev, void* workspace_dev, size_t workspace_bytes,
                                          trtx_stream_t stream);

/* Split form of the fused call (same workspace, same stream order): scan = the HBM-bound streaming
 * kernel alone, then NMS over its tiles.  Used to time the scan kernel in isolation and to overlap the
 * scan of batch i+1 with the NMS of batch i on two streams. */
TRTX_API int trtx_yolo_scan_enqueue(const trtx_yolo_params* p, int batch, const void* const* inputs_dev,
                                    void* workspace_dev, size_t workspace_bytes, trtx_stream_t stream);
TRTX_API int trtx_yolo_nms_after_scan_enqueue(const trtx_yolo_params* p, const trtx_nms_params* q, int batch,
                                              const void* const* inputs_dev, float* compact_out_dev,
                                              int32_t* keep_index_dev, void* workspace_dev, size_t workspace_bytes,
                                              trtx_stream_t stream);

/* Multi-GPU gather of the compact detections over NVLink peer memory (SURVEY 8e: images shard by batch, the only exchange is
 * this gather).  One process per GPU on one NVSwitch node; every rank owns
 *   out   : [slots][world*batch][1 + max_det*R] fp32  -- the gathered detections (rank r's images at [r*batch, (r+1)*batch))
 *   flags : [world][slots] uint32, zero-initialised   -- flags[r][s] = how often rank r has published slot s
 *   ctrl  : [4] uint32, zero-initialised, local only  -- [1] scratch counter, [2] error (1 = a wait timed out)
 * allocated with trtx_peer_alloc (cudaMalloc + CUDA IPC handle) and mapped into the other ranks with trtx_peer_open, so
 * that out_dev[] / flags_dev[] hold, on every rank, the addresses of all ranks' buffers ([rank] = its own).  `slot` is chosen
 * by the caller per call (plain data: calls captured into CUDA graphs keep their slot).
 *   PUBLISH  trtx_gather_push_enqueue: gather_copy_kernel (one CTA per image) copies the live part [count, rows] of every image
 *            of a local compact output into `slot` of EVERY rank's `out` (lane-consecutive NVLink stores; no fence, no flag), then
 *            gather_publish_kernel (one warp) raises this rank's counter of the slot on every rank with relaxed system-scope
 *            stores: the kernel boundary between the two orders the rows before the counter, so no thread executes a system-scope
 *            fence.  Neither kernel waits for anybody.
 *            trtx_yolo_decode_nms_gather_enqueue publishes from inside nms_kernel instead (no extra launch; ONE system-scope
 *            fence by the last CTA; the NMS CTAs' 32 whole SMs stay occupied during the copy -- measured in DESIGN.md section 5).
 *   WAIT     trtx_gather_wait_enqueue (one warp, relaxed polls): returns on the stream once every rank's counter of `slot` has
 *            reached this rank's own, i.e. all ranks' rows of this round are in the local out[slot]; LATER work of the stream
 *            (kernels, copies) may read them.  Rows past an image's `count` are stale.  Gives up after ~2 s (ctrl[2] = 1) instead
 *            of hanging the GPU.
 * Reusing a slot overwrites it on every rank: a rank may publish into a slot again only after all ranks have finished
 * reading the previous round.  The pattern that guarantees it without further handshakes: 2*G slots used in halves; the G
 * publishes of a round go to one half, then the G waits, all on the streams of the round; the next round uses the other half.
 * (A rank cannot get two rounds ahead of a peer: its own waits need the peer's publishes of the round in between.)
 * Every rank must enqueue the same sequence.  world <= 8. */
typedef struct trtx_gather {
    int32_t world, rank, slots, slot;
    float* out_dev[8];
    uint32_t* flags_dev[8];
    uint32_t* ctrl_dev;
} trtx_gather;
TRTX_API int trtx_yolo_decode_nms_gather_enqueue(const trtx_yolo_params* p, const trtx_nms_params* q, int batch,
                                                 const void* const* inputs_dev, float* compact_out_dev,
                                                 int32_t* keep_index_dev, void* workspace_dev, size_t workspace_bytes,
                                                 const trtx_gather* gather, trtx_stream_t stream);
TRTX_API int trtx_gather_push_enqueue(const trtx_gather* gather, const float* compact_out_dev, int batch, int max_det,
                                      int extra_floats, trtx_stream_t stream);
TRTX_API int trtx_gather_wait_enqueue(const trtx_gather* gather, trtx_stream_t stream);
/* The same for n <= 8 consecutive slots slot .. slot+n-1 in ONE launch each (a round of n steps: one push kernel publishing
 * the n local outputs compact_outs_dev[0..n) -- a HOST array of device pointers -- with a single expensive release, one wait
 * kernel for the n slots; world * n <= 64).  A publish reads its sources when it runs: keep them unchanged until then (bench.py
 * double-buffers the compact outputs so that the next NMS never has to wait for the publish of the previous one). */
TRTX_API int trtx_gather_push_many_enqueue(const trtx_gather* gather, const float* const* compact_outs_dev, int n, int batch,
                                           int max_det, int extra_floats, trtx_stream_t stream);
TRTX_API int trtx_gather_wait_many_enqueue(const trtx_gather* gather, int nslots, trtx_stream_t stream);
/* Peer-mappable device memory (zero-initialised) + its 64-byte CUDA IPC handle; open / close a peer's handle; free. */
TRTX_API int trtx_peer_alloc(size_t bytes, void** dev_ptr, unsigned char handle[64]);
TRTX_API int trtx_peer_open(const unsigned char handle[64], void** dev_ptr);
TRTX_API int trtx_peer_close(void* dev_ptr);
TRTX_API int trtx_peer_free(void* dev_ptr);

/* =====================================================================================
 * 3. Decode_TRT (RetinaFace) -- replaces retinaface/decode.cu:110-199
 *    inputs_dev[l] : [batch, 32, (in_h/s)*(in_w/s)] fp32, s = 8,16,32, channels [bbox 2x4 | cls 2x2 | lmk 2x10]
 *    output_dev    : [batch, 1 + total_priors*15] fp32, rows x1,y1,x2,y2,conf,lmk[10]
 *    (TRTX_RETINA_ANTICOV: [batch, 38, g] inputs, [batch, 1 + total_priors*16] output)
 * ===================================================================================== */
enum {
    TRTX_RETINA_FACE = 0,    /* retinaface/decode.cu */
    TRTX_RETINA_ANTICOV = 1, /* retinafaceAntiCov/decode.cu:110-172 (SURVEY 8f rank 4): inputs [batch, 38, g] =
                                [cls 4 | bbox 2x4 | lmk 2x10 | type 6], all soft-maxed by the network; rows of 16 floats
                                x1,y1,x2,y2,conf,lmk[10],mask_conf (decode.h:13-18); gate is the literal `conf < 0.5`;
                                the reference decodes batch 1 only, this build every image */
};
typedef struct trtx_retina_params {
    int32_t in_h, in_w; /* decodeplugin::INPUT_H / INPUT_W (compile-time 480x640 in decode.h:16-17) */
    float gate;         /* 0.02 (decode.cu:131); compared as `conf <= gate`.  Unused by TRTX_RETINA_ANTICOV */
    int32_t variant;    /* TRTX_RETINA_FACE (0, what a zeroed struct selects) | TRTX_RETINA_ANTICOV */
} trtx_retina_params;

TRTX_API int trtx_retina_total_priors(const trtx_retina_params* p);
TRTX_API size_t trtx_retina_workspace_size(const trtx_retina_params* p, int batch);
TRTX_API int trtx_retina_decode_enqueue(const trtx_retina_params* p, int batch, const void* const* inputs_dev,
                                        float* output_dev, void* workspace_dev, size_t workspace_bytes,
                                        trtx_stream_t stream);

/* =====================================================================================
 * 4. Faster R-CNN plugins -- same "null workspace returns the size" idiom as the reference
 *    free functions (rcnn/RpnNms.cu:63-80): call with workspace_dev == NULL to get bytes.
 *    All images of the batch are processed in one launch (the reference loops on the host).
 * ===================================================================================== */
/* rpnDecode, rcnn/RpnDecode.cu:27-143.  inputs: scores [B,A,H,W], deltas [B,A*4,H,W];
 * outputs: scores [B,top_n], boxes [B,top_n,4].  anchors_host: A*4 floats (host memory, copied
 * into the launch parameters -- no H2D copy per enqueue). */
TRTX_API int64_t trtx_rpn_decode(int batch, const float* scores_dev, const float* deltas_dev, float* out_scores_dev,
                                 float* out_boxes_dev, int height, int width, int image_height, int image_width,
                                 float stride, const float* anchors_host, int num_anchors, int top_n,
                                 void* workspace_dev, size_t workspace_bytes, trtx_stream_t stream);
/* rpnNms, rcnn/RpnNms.cu:59-121.  inputs: scores [B,pre], boxes [B,pre,4]; output boxes [B,post,4]. */
TRTX_API int64_t trtx_rpn_nms(int batch, const float* scores_dev, const float* boxes_dev, float* out_boxes_dev,
                              int pre_nms_topk, int post_nms_topk, float nms_thresh, void* workspace_dev,
                              size_t workspace_bytes, trtx_stream_t stream);
/* predictorDecode, rcnn/PredictorDecode.cu:24-110.  inputs: scores [B,N,C], deltas [B,N*C,4],
 * proposals [B,N,4]; outputs scores/boxes/classes [B,N,...]. */
TRTX_API int64_t trtx_predictor_decode(int batch, const float* scores_dev, const float* deltas_dev,
                                       const float* proposals_dev, float* out_scores_dev, float* out_boxes_dev,
                                       float* out_classes_dev, int num_boxes, int num_classes, int image_height,
                                       int image_width, const float* bbox_reg_weights_host, void* workspace_dev,
                                       size_t workspace_bytes, trtx_stream_t stream);
/* batchedNms, rcnn/BatchedNms.cu:92-162.  nms_method 0 hard / 1 soft-linear / 2 soft-gaussian. */
TRTX_API int64_t trtx_batched_nms(int nms_method, int batch, const float* scores_dev, const float* boxes_dev,
                                  const float* classes_dev, float* out_scores_dev, float* out_boxes_dev,
                                  float* out_classes_dev, int count, int detections_per_im, float nms_thresh,
                                  void* workspace_dev, size_t workspace_bytes, trtx_stream_t stream);

/* =====================================================================================
 * 5. Pre-process -- batched letterbox warp + BGR->RGB + /255 + HWC->CHW (+fp16)
 *    replaces warpaffine_kernel / cuda_preprocess / cuda_batch_preprocess,
 *    yolov8/src/preprocess.cu:7-127 (one launch + one stream sync PER IMAGE there).
 * ===================================================================================== */
typedef struct trtx_image_desc {
    const uint8_t* data_dev; /* u8 HWC BGR, row pitch = pitch bytes */
    int32_t width, height;
    int32_t pitch; /* bytes per row, >= 3*width */
    int32_t reserved;
} trtx_image_desc;

/* images_host: array of `batch` descriptors in HOST memory (copied into launch parameters);
 * dst_dev: [batch, 3, dst_h, dst_w] fp32 or fp16 (out_dtype TRTX_F32 | TRTX_F16). One launch. */
TRTX_API int trtx_preprocess_batch_enqueue(const trtx_image_desc* images_host, int batch, void* dst_dev, int dst_w,
                                           int dst_h, int out_dtype, trtx_stream_t stream);
/* The reference's d2s matrix (preprocess.cu:98-110): scale, centre, cv::invertAffineTransform. */
TRTX_API void trtx_letterbox_matrix(int src_w, int src_h, int dst_w, int dst_h, float d2s[6]);
/* get_rect (yolov8/src/postprocess.cpp:6-36, yolov5/src/postprocess.cpp:4-29): maps a detection box from network-input
 * pixels back to the original image: rect = {x, y, width, height} as cv::Rect.  variant TRTX_YOLO_V8: box l,t,r,b,
 * result clamped to the image; TRTX_YOLO_V5: box cx,cy,w,h.  Host function (no device work). */
TRTX_API int trtx_get_rect(int variant, int net_w, int net_h, int img_w, int img_h, const float bbox[4], int rect[4]);

/* get_rect_adapt_landmark (yolov8/src/postprocess.cpp:38-69): like get_rect for the pose models -- the box (l,t,r,b) becomes
 * a cv::Rect in the original image and the num_kpts keypoints (x, y, conf triplets, `lmk`) are mapped IN PLACE.  Host function. */
TRTX_API int trtx_get_rect_adapt_landmark(int net_w, int net_h, int img_w, int img_h, const float bbox[4], float* lmk,
                                          int num_kpts, int rect[4]);
/* RetinaFace's own get_rect_adapt_landmark (retinaface/common.hpp:65-89): 5 landmarks as x, y pairs, modified in place; the box
 * corners are truncated to int and not clamped; rect = {x, y, w, h} in the original image. */
TRTX_API int trtx_retina_get_rect_adapt_landmark(int input_w, int input_h, int img_w, int img_h, const float bbox[4], float lmk[10],
                                                 int rect[4]);
/* process_decode_ptr_host (yolov8/src/postprocess.cpp:131-147): rows of a compact buffer [1 + K*bbox_element] (the output
 * of the ONESHOT mode / cuda_decode+cuda_nms) whose keep flag is 1 -> 6-float rows l,t,r,b,conf,cls.  Returns the number
 * of rows written (<= count), or a negative TRTX_ERR_*.  Host function on HOST memory. */
TRTX_API int trtx_process_decode_ptr_host(const float* decode_ptr_host, int bbox_element, int count, float* rows_out);
/* process_decode_ptr_host_obb (:273-290): rows_out gets 7 floats per kept row (l/cx, t/cy, r/w, b/h, conf, class, angle = column 7 of
 * the 8-float rows of the oriented-box decode); bbox_element >= 8. */
TRTX_API int trtx_process_decode_ptr_host_obb(const float* decode_ptr_host, int bbox_element, int count, float* rows_out);
/* scale_mask (yolov8/src/postprocess.cpp:207-226): the letterboxed region of a network-size mask, resized (cv::resize,
 * bilinear) to the original image.  trtx_scale_mask_rect = the crop rectangle {x, y, w, h} (host);
 * trtx_scale_mask_enqueue: masks_dev [n, net_h, net_w] fp32 -> out_dev [n, img_h, img_w] fp32, one launch, HBM-write-bound. */
TRTX_API int trtx_scale_mask_rect(int net_w, int net_h, int img_w, int img_h, int rect[4]);
TRTX_API int trtx_scale_mask_enqueue(const float* masks_dev, int n, int net_w, int net_h, int img_w, int img_h, float* out_dev,
                                     trtx_stream_t stream);

/* RoIAlign and MaskRcnnInference (SURVEY 8f rank 2): replace roiAlign (rcnn/RoiAlign.cu:150-183) and maskRcnnInference
 * (rcnn/MaskRcnnInference.cu:35-63); same argument meaning, whole batch in one launch, no cudaDeviceSynchronize().
 * rois_dev [batch, num_proposals, 4] x1,y1,x2,y2; features_dev [batch, out_channels, feature_h, feature_w];
 * out_dev [batch, num_proposals, out_channels, pooler_resolution, pooler_resolution].  sampling_ratio <= 0: adaptive. */
TRTX_API int trtx_roi_align(int batch, const float* rois_dev, const float* features_dev, float* out_dev, int pooler_resolution,
                            float spatial_scale, int sampling_ratio, int num_proposals, int out_channels, int feature_h,
                            int feature_w, trtx_stream_t stream);
/* The same with the kernel chosen by the caller (both are bit-identical to the reference's roiAlign):
 * TRTX_ROI_WINDOW (what trtx_roi_align uses) stages each proposal's feature-map window in shared memory and takes the
 * bilinear taps from there -- for the reference's configuration class: pooler_resolution 14, out_channels % 4 == 0,
 * feature_h * feature_w <= 4096; any other shape runs TRTX_ROI_DIRECT, which takes every tap from global memory (the
 * round-1 kernel). */
#define TRTX_ROI_WINDOW 0
#define TRTX_ROI_DIRECT 1
TRTX_API int trtx_roi_align_ex(int batch, const float* rois_dev, const float* features_dev, float* out_dev, int pooler_resolution,
                               float spatial_scale, int sampling_ratio, int num_proposals, int out_channels, int feature_h,
                               int feature_w, int mode, trtx_stream_t stream);
/* indices_dev [batch, detections_per_im] class index as float; masks_dev [batch, detections_per_im, num_classes, S, S];
 * out_dev [batch, detections_per_im, S, S] = sigmoid of the predicted class' mask (rows with an index outside
 * [0, num_classes) are left untouched, as in the reference). */
TRTX_API int trtx_mask_rcnn_inference(int batch, const float* indices_dev, const float* masks_dev, float* out_dev,
                                      int detections_per_im, int output_size, int num_classes, trtx_stream_t stream);

/* The INT8 calibrator's host pre-process (SURVEY 8f rank 4): Int8EntropyCalibrator2::getBatch, yolov8/src/calibrator.cpp:33-52
 * = preprocess_img (yolov8/include/utils.h:6-26: cv::resize INTER_LINEAR of the 8-bit image into the letterbox rectangle, 128-grey
 * canvas) + cv::dnn::blobFromImages(1 / 255.0, swapRB).  HOST code, like the reference's (calibration is not in the inference loop):
 * bgr = 8-bit BGR rows of src_pitch bytes; out_chw = [3, net_h, net_w] fp32 RGB planes, ready for the cudaMemcpy of :48.  The
 * OpenCV arithmetic is restated (fixed-point bilinear resize, float scale) and pinned bit for bit against cv2 4.13.
 * trtx_calib_letterbox_rect: the rectangle {x, y, w, h} the resized image occupies. */
TRTX_API int trtx_calib_letterbox_rect(int src_w, int src_h, int net_w, int net_h, int rect[4]);
TRTX_API int trtx_calib_letterbox_host(const uint8_t* bgr, int src_w, int src_h, size_t src_pitch, int net_w, int net_h, float* out_chw);

/* =====================================================================================
 * 6. Instance masks of the segmentation models (SURVEY 8f rank 1)
 *    replaces the HOST function process_mask(), yolov8/yolov8_seg.cpp:17-60 and
 *    yolov5/src/postprocess.cpp:94-125: sigmoid(coeffs . prototypes) inside the detection's
 *    down-scaled rectangle, then cv::resize (bilinear) to the network input size.
 * ===================================================================================== */
typedef struct trtx_mask_params {
    int32_t variant;      /* TRTX_YOLO_V8: rect from (x, y, w, h) with int() truncation and clamping (yolov8_seg.cpp:17-34);
                             TRTX_YOLO_V5: rect from (cx, cy, w, h) with round() (yolov5 postprocess.cpp:94-104) */
    int32_t net_w, net_h; /* kInputW, kInputH: size of the masks written */
    int32_t mask_w, mask_h; /* prototype resolution; must be net/4 like the reference */
    int32_t num_coeffs;   /* 32 */
    int32_t row_floats;   /* floats per detection row of `dets_dev` */
    int32_t coeff_offset; /* first mask coefficient inside a row (box = floats 0..3) */
    int32_t max_masks;    /* masks written per image: the first min(count, max_masks) rows */
} trtx_mask_params;

/* proto_dev: [batch, num_coeffs, mask_h, mask_w] fp32 (the engine's "proto" output);
 * dets_dev : [batch, 1 + max_rows*row_floats] fp32 = count, rows (e.g. the compact NMS output with
 *            extra_floats = 32, extra_offset = 6: row_floats = 39, coeff_offset = 7);
 * masks_dev: [batch, max_masks, net_h, net_w] fp32; slots >= count are left untouched.  One launch. */
TRTX_API int trtx_process_mask_enqueue(const trtx_mask_params* p, int batch, const float* proto_dev, const float* dets_dev,
                                       int max_rows, float* masks_dev, trtx_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TRTX_HOT_H */
