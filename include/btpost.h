/*
 * btpost.h -- C ABI of libbtpost, the sm_100a post-processing + evaluation hot path for
 * multitask bone-tumor YOLO heads.
 *
 * The reference (rafifmalikdzaki/Multitask-Bonetumor-yolo) has no FFI: the path is inline eager
 * PyTorch inside `MultiTaskLitModel.validation_step` (src/running_main_v2.py:643-945) and the
 * intended method `_prepare_det_outputs_for_metrics_and_logging` (src/evaluate_model.py:174-178).
 * Each entry point below names the reference statements it replaces.  Everything is plain C:
 * pointers, sizes, POD structs; no torch types.  All pointers are DEVICE pointers owned by the
 * caller unless stated otherwise.  The library never allocates device memory, never synchronises, and orders
 * all work on the caller's stream (CUDA-graph capturable).  Host-side state: btpost_run borrows a helper stream
 * + five events from a small per-device pool that is created lazily and guarded by a mutex (see btpost_run);
 * nothing else is kept between calls.
 *
 * Return value: 0 on success, a negative BT_ERR_* otherwise (btpost_error_string decodes it).
 */
#ifndef BTPOST_H_
#define BTPOST_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BTPOST_VERSION 100 /* 0.1.0 */
#define BTPOST_API __attribute__((visibility("default")))

enum {
    BT_OK = 0,
    BT_ERR_BAD_ARG = -1,       /* null pointer / non-positive size / inconsistent params */
    BT_ERR_UNSUPPORTED = -2,   /* shape outside what the kernels implement */
    BT_ERR_WORKSPACE = -3,     /* workspace smaller than btpost_workspace_bytes() */
    BT_ERR_MISALIGNED = -4,    /* pointer not aligned as documented */
    BT_ERR_CUDA = -5,          /* a CUDA launch failed; cudaGetLastError text via error_string */
    BT_ERR_NCCL = -6
};

/* Number of COCO area ranges (all, small, medium, large) -- SURVEY.md A.3. */
#define BT_NUM_AREA 4
#define BT_MAX_IOU_THRS 16
#define BT_MAX_CLASSES 16

enum { BT_LAYOUT_L2 = 0, BT_LAYOUT_L1 = 1 };
enum { BT_CLASS_AGNOSTIC = 0, BT_CLASS_AWARE = 1, BT_CLASS_OFFSET = 2 };
enum { BT_GT_LITERAL = 0, BT_GT_INTENDED = 1 };
enum { BT_MASK_U8 = 0, BT_MASK_F32 = 1 };
enum { BT_PROTO_F32 = 0, BT_PROTO_BF16 = 1 };
enum { BT_HEAD_F32 = 0, BT_HEAD_BF16 = 1 };

/* Problem description.  Mirrors the reference's module constants CONF_TH / NMS_IOU / TOP_K
 * (src/running_main_v2.py:51-53) and hparams img_size / nc_det / proto_ch / iou_match_thresh
 * (src/running_main_v2.py:150-188). */
typedef struct BtParams {
    int32_t batch;            /* B images in this call                                        */
    int32_t num_anchors;      /* N (8400 @640^2, 21504 @1024^2)                               */
    int32_t nc;               /* detection classes (<= BT_MAX_CLASSES)                        */
    int32_t nm;               /* mask coefficients / prototype channels (must be 32)          */
    int32_t reg_max;          /* DFL bins (L1 layout only; 16)                                */
    int32_t img_h, img_w;     /* network input size S                                         */
    int32_t proto_h, proto_w; /* prototype resolution; must equal img/4                       */
    int32_t layout;           /* BT_LAYOUT_L2: head [B,4+nc+nm,N]; BT_LAYOUT_L1: 3 raw maps   */
    float conf_thres;         /* CONF_TH, strict >                                            */
    double iou_thres;         /* NMS_IOU (torchvision takes a double)                         */
    int32_t max_det;          /* TOP_K                                                        */
    int32_t max_cand;         /* Ultralytics max_nms: when more than max_cand anchors pass the filter only the
                                 max_cand best-scoring ones (stable: ties -> lower anchor index) enter the NMS;
                                 0 => no limit.  n_cand still reports every anchor that passed the filter and
                                 det_keep still indexes that full (anchor-ordered) list.                      */
    int32_t class_mode;       /* BT_CLASS_*; reference = agnostic                             */
    float max_wh;             /* class offset for BT_CLASS_OFFSET (Ultralytics 7680)          */
    int32_t clamp_boxes;      /* clamp_(0, img) after the filter (reference: 1)               */
    int32_t gt_mode;          /* BT_GT_LITERAL reproduces cat(...).view(-1,4) as shipped      */
    int32_t max_gt;           /* GT capacity per image (<= 32); rows beyond it are dropped and reported
                                 through BtIO.gt_overflow (the reference has no limit)                       */
    int32_t num_gt_rows;      /* rows of det_boxes_gt [G_total, 6]                            */
    float iou_match_thresh;   /* anchor<->GT confusion-matrix matching threshold (0.5)        */
    int32_t crop;             /* crop instance masks to their box at prototype resolution     */
    int32_t gt_mask_dtype;    /* BT_MASK_U8 or BT_MASK_F32 (reference dataset dtype)          */
    float proj_bias;          /* bias of seg_proto_projector Conv2d(nm->1,k=1)                */
    int32_t num_iou_thrs;     /* T (10 for mAP50-95, 1 for mAP50)                             */
    double iou_thrs[BT_MAX_IOU_THRS]; /* float64(fp32 linspace(0.5,0.95,10))                  */
    int32_t image_offset;     /* global index of image 0 of this batch: written into the sweep records (BtIO.sweep)
                                 so that the AP order does not depend on the sharding                         */
    int32_t nms_threads;      /* threads per image of the NMS kernel: 0 = default (1024), 512 (small footprint: several batches in flight), 256, 1024 */
    int32_t proto_dtype;      /* BT_PROTO_F32 (default) or BT_PROTO_BF16: dtype of `protos`; bf16 values are widened exactly, so the
                                 results equal those of the reference on `protos.float()` (it validates under bf16-mixed) */
    int32_t head_dtype;       /* BT_HEAD_F32 (default) or BT_HEAD_BF16: dtype of the L2 `head` / the L1 raw maps + coeffs (same exact widening) */
    int32_t drop_gt_no_cand;  /* 1 = v2 behaviour (running_main_v2.py:797-814): an image in which no anchor passes
                                 CONF_TH gets an EMPTY target, i.e. its GT boxes leave the mAP denominator;
                                 0 = v3 behaviour (running_main_v3.py:541-571): the target is kept             */
    int32_t in_flight;        /* batches the caller keeps in flight on this device (btpost.Pipeline: its depth).  0 / 1: the
                                 persistent kernels of the mask stage size their grids for a GPU of their own (4 / 8 CTAs per
                                 SM); >= 2: for a shared one (3 / 6: other batches' CTAs find room beside them, measured
                                 -1.5 % per pipelined step).  Results do not depend on it.                              */
    int32_t io_soft_dice;     /* 0: `io` points to a BtIO; 1: to a BtIOSoftDice (a BtIO followed by the soft-Dice outputs) */
    union {                   /* io_micro took the former reserved word: the size and every offset are unchanged      */
        int32_t io_micro;     /* 1: `io` points to a BtIOMicro (a BtIOSoftDice followed by micro_sweep); its soft-Dice pointers
                                 are then read whatever io_soft_dice says (NULL skips them).  0: see io_soft_dice        */
        int32_t reserved[1];
    };
} BtParams;

/* Device buffers.  Inputs are read-only.  Any OUTPUT pointer may be NULL to skip that output
 * unless marked required.  Shapes use B=batch, N=num_anchors, K=max_det, G=max_gt, S=img,
 * A=BT_NUM_AREA, T=num_iou_thrs. */
typedef struct BtIO {
    /* ---- inputs ---- */
    const void *head;           /* L2: [B, 4+nc+nm, N] fp32 or bf16 (head_dtype) (segment_preds_cat, main_modelv2.py:367),
                                   16-byte aligned; N <= 32768, or N <= 8192 when N % 4 != 0 (L1: N <= 32768)      */
    const void *maps[3];        /* L1: [B, 4*reg_max+nc, H_l, W_l], strides 8/16/32; fp32 or bf16 (head_dtype) */
    const void *coeffs;         /* L1: mask coefficients [B, nm, N] (Segment `mc`), same dtype as the maps   */
    const void *protos;         /* [B, nm, proto_h, proto_w] fp32 (or bf16: proto_dtype), 16-byte aligned */
    const float *det_boxes_gt;  /* [num_gt_rows, 6] (batch_idx, cls, cx, cy, w, h) normalised  */
    const void *masks_gt;       /* [B, 1, S, S] u8 or f32 {0,1}                                */
    const float *proj_weight;   /* [nm] seg_proto_projector weight                             */
    /* ---- detection outputs (required) ---- */
    int32_t *det_count;         /* [B]                                                         */
    float *dets;                /* [B, K, 6] xyxy, score, float(label)   (a5 `[K,6]`)          */
    int64_t *det_keep;          /* [B, K] NMS keep indices into the filtered list (int64)      */
    int32_t *det_anchor;        /* [B, K] original anchor index                                */
    float *det_coeff;           /* [B, K, nm] mask coefficients of kept detections             */
    int32_t *n_cand;            /* [B] candidates that passed the filter                       */
    /* ---- GT outputs (required) ---- */
    int32_t *gt_count;          /* [B]                                                         */
    float *gt_boxes;            /* [B, G, 4] clamped xyxy (mAP copy, running_main_v2.py:849-865) */
    float *gt_boxes_raw;        /* [B, G, 4] unclamped xyxy (loss copy, :409-433)              */
    int32_t *gt_labels;         /* [B, G]                                                      */
    /* ---- metric accumulators (ACCUMULATED: caller zeroes them at sweep start) ---- */
    int64_t *cm;                /* [nc, nc] confusion counts [gt][pred]  (a10)                 */
    int64_t *seg_cnt4;          /* [4] tp, fp, fn, tn of the projector mask (a8 i)             */
    int64_t *uni_cnt4;          /* [4] same for the union of instance masks                    */
    /* ---- per-batch metric outputs ---- */
    int32_t *cm_pos;            /* [B] positive anchors per image                              */
    int64_t *seg_img3;          /* [B, 3] inter, |P|, |G| for the projector mask (a8 ii,iii)   */
    float *seg_dice;            /* [B]                                                         */
    float *seg_iou;             /* [B]                                                         */
    int64_t *uni_img3;          /* [B, 3] same for the union of instance masks                 */
    float *uni_dice;            /* [B]                                                         */
    float *uni_iou;             /* [B]                                                         */
    int32_t *inst_area;         /* [B, K] pixels of each instance mask                         */
    int32_t *inst_inter;        /* [B, K] pixels of each instance mask inside the GT mask      */
    /* ---- optional dense outputs ---- */
    uint8_t *seg_mask;          /* [B, S, S] projector mask (seg_preds, running_main_v2.py:703) */
    float *seg_logits;          /* [B, S, S] upsampled projector logits (seg_logits_for_logging) */
    uint8_t *uni_mask;          /* [B, S, S] union of instance masks                           */
    uint8_t *inst_bits;         /* [B, K, S, S/8] every instance mask, bit-packed: bit (x & 7) of byte x >> 3 of row y
                                   (numpy packbits, bitorder="little"); planes k >= det_count[b] are zero.
                                   src/test_model.py:80-85 (einsum -> bilinear -> sigmoid > 0.5) with the Ultralytics
                                   crop (BtParams.crop).  16-byte aligned                                            */
    uint8_t *inst_masks;        /* [B, K, S, S] the same masks as bytes {0,1} (the reference's bool tensor); needs
                                   inst_bits as well (the bytes are expanded from the bits).  16-byte aligned        */
    /* ---- COCO matching outputs (a9) ---- */
    int32_t *dt_match;          /* [B, A, T, K] matched GT index + 1, 0 = unmatched            */
    uint8_t *dt_ignore;         /* [B, A, T, K]                                                */
    uint8_t *gt_ignore;         /* [B, A, G]                                                   */
    /* ---- optional: v3 segmentation-mAP prep (a11, src/running_main_v3.py:478-498) ---- */
    double *seg_prob_sum;       /* [B] sum of sigmoid(logit) over the projector mask's foreground pixels:
                                   score = seg_prob_sum / (|P| + 1e-6); |P|, mask IoU from seg_img3     */
    /* ---- optional ---- */
    int32_t *gt_rows_total;     /* [B] rows of det_boxes_gt that belong to the image BEFORE the max_gt cut: a value
                                   above max_gt means GT rows were dropped (the host wrapper raises)     */
    void *sweep;                /* sweep state (btpost_sweep_*): per-detection AP records, GT counts, image count and
                                   Dice / IoU sums of this batch are appended on the device (needs dt_match, dt_ignore,
                                   gt_ignore)                                                            */
    const int32_t *image_base;  /* [1] optional, device: added to BtParams.image_offset when the records are written, so
                                   that a step captured into a CUDA graph can be replayed for different batches  */
    void *seg_sweep;            /* optional sweep state (same format as `sweep`, 16-byte aligned) for the v3 segmentation mAP
                                   (a11, src/running_main_v3.py:478-498): finalize_kernel appends ONE record per image -- the
                                   projector mask scored by its mean foreground probability against the GT mask, class 0.
                                   Needs seg_img3 and seg_prob_sum.  Record fields:
                                     matched / ignored  bit a * T + t: mask IoU >= min(iou_thrs[t], 1 - 1e-10); ignored = matched ?
                                                        |G| outside area range a : |P| outside area range a (COCOeval)
                                     score_key          desc_key(seg_prob_sum / (|P| + 1e-6)), fp32 as the reference computes it
                                     image              BtParams.image_offset + *image_base + index in the batch
                                     rank = class_rank = label = 0
                                   Header: N_RECORDS, N_IMAGES, NPIG[a][0] (|G| inside area range a); the FSUM slots stay
                                   unused.  btpost_sweep_accumulate with nc = 1, max_det_per_image = 1 gives the tables. */
} BtIO;

/* v3 soft Dice of the projector probabilities (SURVEY.md A.4, src/running_main_v3.py:466-474): a BtIO followed by three
 * optional outputs.  Pass a pointer to it as the `io` of every entry point, with BtParams.io_soft_dice = 1; BtIO itself
 * keeps its layout.  p = 1 / (1 + exp(-x)) of every upsampled projector logit x (the oracle's fma-only exp, IEEE
 * division; p = 0 for x < -87), t = the GT mask.  Each p is rounded to 2^-40 fixed point, so the sums do not depend on
 * the order of the atomics. */
typedef struct BtIOSoftDice {
    BtIO io;
    int64_t *seg_soft2;         /* [B, 2] sum of p * t and sum of p over the S^2 pixels, units of 2^-40; zeroed per call by
                                   the NMS stage (like seg_prob_sum)                                                    */
    float *seg_soft_dice;       /* [B] 2 A / (P + G) in double rounded to fp32 (A, P from seg_soft2, G = |G|); NaN when
                                   P + G == 0.  Needs seg_soft2                                                         */
    int64_t *seg_soft_acc;      /* [2] ACCUMULATED like cm / seg_cnt4: sum over images of round(soft Dice * 2^40), and the
                                   number of images with a defined soft Dice.  Needs seg_soft2                          */
} BtIOSoftDice;

/* Class-agnostic box mAP (torchmetrics MeanAveragePrecision(average="micro"), which sets every prediction and target label
 * to 0 before the COCO evaluation): a BtIOSoftDice followed by a third sweep state.  Pass a pointer to it as the `io` of
 * every entry point, with BtParams.io_micro = 1; BtIO and BtIOSoftDice keep their layouts. */
typedef struct BtIOMicro {
    BtIOSoftDice sd;
    void *micro_sweep;          /* optional sweep state (same format as BtIO.sweep, 16-byte aligned; needs dt_match): match_kernel
                                   runs COCOeval.evaluateImg a second time per image with the labels ignored -- one category,
                                   every kept detection in its descending-score order, every GT of the image, the same area
                                   ranges, IoU thresholds and ignore rules -- on the IoUs of the class-aware pass, and appends
                                   ONE record per kept detection.  The class-aware outputs do not depend on it.  Record fields:
                                     matched / ignored  bit a * T + t, from the class-agnostic matching
                                     score_key, image, rank   as in BtIO.sweep
                                     class_rank = rank  (the maxDets cut is per image: greedy matching in score order means
                                                        that the cut only drops records, so matching all K and cutting in
                                                        the accumulate is exact)
                                     label = 0
                                   Header: N_RECORDS, N_IMAGES, NPIG[a][0] (non-ignored GTs of every class in area range a;
                                   drop_gt_no_cand removes them as it does for BtIO.sweep); the FSUM slots stay unused.
                                   btpost_sweep_accumulate with nc = 1, max_det_per_image = max_det gives the tables. */
} BtIOMicro;

/* Library / build identification. */
BTPOST_API int btpost_version(void);
BTPOST_API const char *btpost_error_string(int code);
/* Fills *bytes with the workspace size btpost_* calls need for `p` (256-byte aligned pointer). */
BTPOST_API int btpost_workspace_bytes(const BtParams *p, size_t *bytes);

/* Stage entry points.  They share one workspace layout, so they may be called in sequence on
 * the same stream (decode_filter -> nms_match -> masks) or through btpost_run. */

/* a2+a3+a6+a10: box decode, max/argmax over classes, strict conf filter, clamp, ordered
 * compaction; GT prep; anchor<->GT confusion-matrix matching.
 * Replaces src/running_main_v2.py:743-795, :842-882, :402-449,:476-486 (+ batch_bbox_iou :68-94). */
BTPOST_API int btpost_decode_filter(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream);

/* a4+a5+a9(match): stable descending sort, greedy NMS with early exit at max_det (keeps are
 * bit-exact against torchvision.ops.nms(...)[:TOP_K]), gather of kept detections, COCOeval
 * evaluateImg matching.  Replaces src/running_main_v2.py:817-839 and the per-image part of
 * torchmetrics MeanAveragePrecision (:884-892). */
BTPOST_API int btpost_nms_match(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream);

/* a7+a8: projector mask (Conv2d nm->1, bilinear x4, sigmoid>0.5) and instance masks
 * (coeff . protos, crop, bilinear x4, sigmoid>0.5), pixel counters, per-image Dice / IoU.
 * Replaces src/running_main_v2.py:689-713, src/test_model.py:15-23,80-89. */
BTPOST_API int btpost_masks(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream);

/* The kernels of btpost_masks one by one (same arguments; `parts` is an OR of BT_MASKS_*), in the order
 * PACK -> CONTRACT -> CELLS on one stream: GT mask bytes -> bits (independent of the detections), the one pass over
 * the prototypes (projector + per-detection K=32 contraction, logits to the workspace), bilinear x4 + threshold +
 * counters + per-image Dice/IoU.  Used by btpost_run to overlap PACK with the detection stages, and by bench.py to
 * time the HBM-side kernel alone. */
enum { BT_MASKS_PACK = 1, BT_MASKS_CONTRACT = 2, BT_MASKS_CELLS = 4 };
BTPOST_API int btpost_masks_parts(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream, int parts);

/* Whole hot path for one batch: the three stages above, ordered on `stream`.  The GT-bit packing and the COCO
 * matching run on a helper stream of the library that is forked from and joined back into `stream` with events, so
 * the call is still a unit of work on `stream` and capturable into a CUDA graph.  Every call borrows its (helper stream,
 * events) set from a mutex-guarded per-device pool: concurrent calls from several host threads are safe as long as
 * they use different workspaces / output buffers (two calls that share a workspace must be ordered by the caller). */
BTPOST_API int btpost_run(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream);

/* Binned precision-recall / ROC state of the projector probabilities (torchmetrics BinaryPrecisionRecallCurve / BinaryROC /
 * BinaryAUROC / BinaryAveragePrecision with thresholds=T; DESIGN.md §4).  Every one of the S^2 pixels of every image counts:
 * p = 1 / (1 + exp(-x)) of its upsampled projector logit x exactly as soft Dice computes it (BtIOSoftDice; p = 0 for
 * x < -87), t = its GT bit (the one seg_cnt4 counts).  A pixel is predicted positive at threshold k iff p >= thr[k]; a NaN
 * p is below every threshold.
 *
 * PRECONDITION: enqueued after btpost_masks or btpost_run on the same workspace, stream and BtParams.  It reads the
 * projector logits [B, proto_h, proto_w] and the GT block words those calls leave in the workspace, so no other call may
 * use the workspace in between.
 *
 * `thresholds` [num_thresholds] is a HOST array: fp32 values in [0, 1], non-decreasing, 2 <= num_thresholds <=
 * BT_MAX_CURVE_THRS (torchmetrics' thresholds=T is the fp32 linspace(0, 1, T)); it is copied into the launch.
 * `hist` [2, num_thresholds + 1] int64 (device, 8-byte aligned) is ACCUMULATED like seg_cnt4: hist[t][j] += pixels with GT
 * bit t and exactly j thresholds <= p.  Confusion counts at threshold k: tp = sum_{j>k} hist[1][j], fp = sum_{j>k}
 * hist[0][j], fn = sum_{j<=k} hist[1][j], tn = sum_{j<=k} hist[0][j].  Integer sums: the words do not depend on the launch
 * shape, the order or the batch composition.  Arguments are checked before any CUDA call. */
#define BT_MAX_CURVE_THRS 1024
BTPOST_API int btpost_seg_curve(const BtParams *p, void *ws, size_t ws_bytes, const float *thresholds, int32_t num_thresholds,
                                int64_t *hist, void *stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Sweep state (a9 accumulate/summarize; replaces torchmetrics MeanAveragePrecision's state lists + COCOeval.accumulate,
 * src/running_main_v2.py:884-892, :1017-1098, src/evaluate_model.py:180-182, :291-319).
 *
 * Caller-owned device memory: BT_SWEEP_HEADER_I64 int64 counters followed by a ring of 32-byte per-detection records.
 * With BtIO.sweep set, btpost_run / btpost_nms_match / btpost_masks append to it on the device (no host work per
 * batch): match_kernel writes one record per kept detection and adds the batch's non-ignored GT counts and image
 * count, finalize_kernel adds the per-image Dice / IoU (2^-40 fixed point, so the sums do not depend on the order of
 * the atomics).  A second state at BtIO.seg_sweep collects the v3 segmentation mAP (one record per image, nc = 1), a third at
 * BtIOMicro.micro_sweep the class-agnostic box mAP (one record per kept detection, nc = 1).
 * Every header slot is a plain sum, so shards are merged by ONE all-reduce(SUM) over the header (the
 * metric-counter all-reduce of the north star) plus one all-gather of the records (AP needs the global score order).
 * The caller may point BtIO.cm / seg_cnt4 / uni_cnt4 into the header's user slots so that they travel with it. */
#define BT_SWEEP_HEADER_I64 512
enum {
    BT_SWEEP_N_RECORDS = 0,  /* records offered so far; the first min(n, capacity) are in the ring, the excess was
                                dropped (the caller sized the ring too small: the host wrapper raises)    */
    BT_SWEEP_N_IMAGES = 2,
    BT_SWEEP_FSUM = 3,       /* [4] sum of seg dice, seg iou, uni dice, uni iou, units of 2^-40           */
    BT_SWEEP_CAPACITY = 7,   /* ring capacity in records (set by btpost_sweep_reset; not a sum)          */
    BT_SWEEP_NPIG = 8,       /* [BT_NUM_AREA][BT_MAX_CLASSES] non-ignored GT boxes per (area range, class) */
    BT_SWEEP_USER = 72       /* [440] free for the caller: cm [nc*nc], seg_cnt4 [4], uni_cnt4 [4], ...    */
};
typedef struct BtSweepRecord {   /* one kept detection */
    uint64_t matched;        /* bit a * T + t: matched to a GT at area range a, IoU threshold t (dt_match != 0) */
    uint64_t ignored;        /* same indexing: COCOeval dtIgnore                                        */
    uint32_t score_key;      /* order-preserving image of the fp32 score: ascending key = descending score */
    uint32_t image;          /* BtParams.image_offset + index in the batch                               */
    uint16_t rank;           /* position in the image's detection list (descending score)                */
    uint16_t class_rank;     /* earlier detections of the same class in the image (maxDets cut)          */
    uint8_t label;
    uint8_t pad[3];
} BtSweepRecord;

BTPOST_API int btpost_sweep_bytes(int64_t max_records, size_t *bytes);
/* Zeroes the header and sets the capacity (async on `stream`). */
BTPOST_API int btpost_sweep_reset(void *sweep, int64_t max_records, void *stream);

/* COCOeval.accumulate on the device: stable LSD radix sort of the records by (class, score desc, image, rank) -- the
 * order pycocotools gets from concatenating images in order + mergesort on -score -- then, per (class, maxDet, area,
 * IoU threshold), running tp / fp counts and the 101-point interpolated precision (right-to-left running max of
 * tp / (tp + fp + eps), looked up at the first position whose recall reaches each recall threshold) and the final
 * recall.  `records` [n_records] (device; reordered in place), `npig` = header slot BT_SWEEP_NPIG of the merged
 * header (device), `rec_thrs` [num_rec] doubles (device; numpy.linspace(0, 1, 101) for COCO), `max_dets` [num_max_dets]
 * host ints (<= 4), `num_images` bounds BtSweepRecord.image (number of radix passes).  Outputs (device, doubles, the
 * pycocotools layout): precision [T, num_rec, nc, BT_NUM_AREA, num_max_dets], recall [T, nc, BT_NUM_AREA, num_max_dets],
 * -1 where a class has no non-ignored GT.  `scratch` from btpost_sweep_accumulate_bytes (256-byte aligned). */
BTPOST_API int btpost_sweep_accumulate_bytes(int64_t n_records, size_t *bytes);
BTPOST_API int btpost_sweep_accumulate(void *records, int64_t n_records, const int64_t *npig, const double *rec_thrs,
                                       int32_t num_rec, int32_t nc, int32_t num_iou_thrs, const int32_t *max_dets,
                                       int32_t num_max_dets, int32_t max_det_per_image, int64_t num_images,
                                       double *precision, double *recall, void *scratch, size_t scratch_bytes,
                                       void *stream);
/* btpost_sweep_accumulate plus COCOeval.accumulate's third table (NULL skips it): `scores` [T, num_rec, nc, BT_NUM_AREA,
 * num_max_dets] (device, doubles, the layout of `precision`) = the fp32 score, widened, of the first record of the
 * (class, area range, maxDet) sequence -- the class's records with class_rank < maxDet, ignored ones included, in sort
 * order -- whose recall reaches recall threshold r (for r = 0: the sequence's first record, whatever its match / ignore
 * state); 0 when no record reaches it (an empty sequence included); -1 where the class has no non-ignored GT.  This is
 * the score at which pycocotools reaches each recall: how an operating point is chosen. */
BTPOST_API int btpost_sweep_accumulate_ext(void *records, int64_t n_records, const int64_t *npig, const double *rec_thrs,
                                           int32_t num_rec, int32_t nc, int32_t num_iou_thrs, const int32_t *max_dets,
                                           int32_t num_max_dets, int32_t max_det_per_image, int64_t num_images,
                                           double *precision, double *recall, double *scores, void *scratch,
                                           size_t scratch_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Surface distances of a predicted mask against the GT mask: Hausdorff distance, HD95 and ASSD per image, in pixels of
 * the network input (MONAI's compute_hausdorff_distance / compute_average_surface_distance with symmetric ASSD, made
 * exact; DESIGN.md §4).  P = pred != 0, G = gt != 0; edge(M) = M AND NOT erode(M) with the 4-neighbour cross and
 * background outside the image; d = Euclidean distance from each edge pixel of one mask to the nearest edge pixel of the
 * other, computed exactly (integer squared distances, sqrt in double).
 *   hd   = the largest d of both directions
 *   hd95 = max over the two directions of torch.quantile(d.double(), 0.95) (linear interpolation)
 *   assd = mean of the d of both directions together
 * Each is rounded once to fp32.  An image whose P or G is empty gets NaN in all three and is not counted in `acc`.
 * A pure function of the masks: the same bytes whatever else is in the batch.
 *
 * `pred` [B, S, S] bytes (PostProcessor's seg_mask), `gt` [B, 1, S, S] u8 or f32 (gt_mask_dtype), both 16-byte aligned;
 * S % 32 == 0 and S <= 1280.  Outputs hd, hd95, assd [B] (device).  `acc` [4] (device, may be NULL) is ACCUMULATED:
 * sum of round(hd * 2^32), of round(hd95 * 2^32), of round(assd * 2^32) (the fp32 values, widened) over the images with
 * defined values, and their count; integer sums, so the words do not depend on the order of the images.  `scratch` from
 * btpost_surface_bytes (256-byte aligned; 8 * B * S^2 bytes plus 64 * B rounded up to 256).  Arguments are checked before any CUDA call. */
BTPOST_API int btpost_surface_bytes(int32_t batch, int32_t img, size_t *bytes);
BTPOST_API int btpost_surface_distance(int32_t batch, int32_t img, const uint8_t *pred, const void *gt, int32_t gt_mask_dtype,
                                       float *hd, float *hd95, float *assd, int64_t *acc, void *scratch, size_t scratch_bytes,
                                       void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BTPOST_H_ */
