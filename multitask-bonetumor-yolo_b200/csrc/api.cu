// C ABI of libbtpost (declared in include/btpost.h): argument validation + stage dispatch.
#include <math.h>

#include <mutex>
#include <new>

#include "common.cuh"

namespace bt {

static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Anchor limit of the decode/filter kernel: one cluster of 8 CTAs of at most 1024 threads covers an image in one pass.
// The L2 decoder reads 4 anchors per thread when N % 4 == 0 (N <= 8 * 1024 * 4) and 1 otherwise (N <= 8 * 1024); the
// L1 decoder always takes up to 4 anchors per thread, interleaved, whatever N % 4 is.
static int check_anchor_limit(const BtParams *p) {
    const int per_thread = (p->layout == BT_LAYOUT_L1 || p->num_anchors % 4 == 0) ? 4 : 1;
    return p->num_anchors > 8 * 1024 * per_thread ? BT_ERR_UNSUPPORTED : BT_OK;
}

// The problem description alone (btpost_seg_curve takes no BtIO).
static int check_shape(const BtParams *p) {
    if (!p) return BT_ERR_BAD_ARG;
    if (p->batch <= 0 || p->num_anchors <= 0 || p->nc <= 0 || p->max_det <= 0) return BT_ERR_BAD_ARG;
    if (p->nc > BT_MAX_CLASSES || p->nm != 32) return BT_ERR_UNSUPPORTED;
    if (p->max_gt <= 0 || p->max_gt > 32) return BT_ERR_UNSUPPORTED;
    if (p->max_det > 4096) return BT_ERR_UNSUPPORTED;
    if (p->img_h <= 0 || p->img_w <= 0) return BT_ERR_BAD_ARG;
    if (p->proto_h * 4 != p->img_h || p->proto_w * 4 != p->img_w) return BT_ERR_UNSUPPORTED;
    if (p->img_w % 32 != 0 || p->proto_h < 2 || p->proto_w < 2) return BT_ERR_UNSUPPORTED;
    if (p->num_iou_thrs < 0 || p->num_iou_thrs > BT_MAX_IOU_THRS) return BT_ERR_BAD_ARG;
    if (p->num_gt_rows < 0) return BT_ERR_BAD_ARG;
    if (!(p->iou_thres == p->iou_thres)) return BT_ERR_BAD_ARG;
    if (p->nms_threads != 0 && p->nms_threads != 256 && p->nms_threads != 512 && p->nms_threads != 1024) return BT_ERR_BAD_ARG;
    if (p->in_flight < 0) return BT_ERR_BAD_ARG;
    if (p->io_soft_dice != 0 && p->io_soft_dice != 1) return BT_ERR_BAD_ARG;
    if (p->io_micro != 0 && p->io_micro != 1) return BT_ERR_BAD_ARG;
    if (p->proto_dtype != BT_PROTO_F32 && p->proto_dtype != BT_PROTO_BF16) return BT_ERR_BAD_ARG;
    if (p->head_dtype != BT_HEAD_F32 && p->head_dtype != BT_HEAD_BF16) return BT_ERR_BAD_ARG;
    if (p->layout == BT_LAYOUT_L1) {
        if (p->reg_max <= 0 || p->reg_max > 32) return BT_ERR_UNSUPPORTED;
        if (p->img_w % 32 != 0 || p->img_h % 32 != 0) return BT_ERR_UNSUPPORTED;
        int n = 0;
        for (int s = 8; s <= 32; s *= 2) n += (p->img_w / s) * (p->img_h / s);
        if (n != p->num_anchors) return BT_ERR_BAD_ARG;
    } else if (p->layout != BT_LAYOUT_L2) {
        return BT_ERR_BAD_ARG;
    }
    return check_anchor_limit(p);
}

int check_params(const BtParams *p, const BtIO *io) {
    if (!p || !io) return BT_ERR_BAD_ARG;
    return check_shape(p);
}

static int check_ws(const BtParams *p, void *ws, size_t ws_bytes) {
    if (!ws) return BT_ERR_BAD_ARG;
    if (reinterpret_cast<uintptr_t>(ws) & 255) return BT_ERR_MISALIGNED;
    if (ws_bytes < carve(p, nullptr).bytes) return BT_ERR_WORKSPACE;
    return BT_OK;
}

static int check_stage1(const BtParams *p, const BtIO *io) {
    if (p->layout == BT_LAYOUT_L2) {
        if (!io->head) return BT_ERR_BAD_ARG;
        if (!aligned16(io->head)) return BT_ERR_MISALIGNED;   // the decoder reads 4 anchors of a row with one vector load
    } else {
        if (!io->maps[0] || !io->maps[1] || !io->maps[2]) return BT_ERR_BAD_ARG;
    }
    if (p->num_gt_rows > 0 && !io->det_boxes_gt) return BT_ERR_BAD_ARG;
    if (!io->n_cand || !io->gt_count || !io->gt_boxes || !io->gt_boxes_raw || !io->gt_labels || !io->cm || !io->cm_pos)
        return BT_ERR_BAD_ARG;
    return BT_OK;
}

static int check_stage2(const BtParams *p, const BtIO *io) {
    if (!io->n_cand || !io->det_count || !io->dets || !io->det_keep || !io->det_anchor || !io->det_coeff)
        return BT_ERR_BAD_ARG;
    if (p->layout == BT_LAYOUT_L2 ? !io->head : !io->coeffs) return BT_ERR_BAD_ARG;
    if (io->dt_match && (!io->gt_count || !io->gt_boxes || !io->gt_labels || p->num_iou_thrs <= 0)) return BT_ERR_BAD_ARG;
    if (io->sweep && !io->dt_match) return BT_ERR_BAD_ARG;   // the records are written by the COCO matching
    if (io->sweep && (reinterpret_cast<uintptr_t>(io->sweep) & 15)) return BT_ERR_MISALIGNED;
    if (void *ms = micro_sweep_of(*p, *io)) {
        if (!io->dt_match) return BT_ERR_BAD_ARG;   // the class-agnostic pass runs inside the COCO matching
        if (!aligned16(ms)) return BT_ERR_MISALIGNED;
    }
    return BT_OK;
}

static int check_stage3(const BtParams *p, const BtIO *io) {
    if (!io->protos || !io->masks_gt || !io->proj_weight || !io->dets || !io->det_count || !io->det_coeff)
        return BT_ERR_BAD_ARG;
    if (!aligned16(io->protos) || !aligned16(io->masks_gt)) return BT_ERR_MISALIGNED;
    if ((io->seg_mask && !aligned16(io->seg_mask)) || (io->uni_mask && !aligned16(io->uni_mask))) return BT_ERR_MISALIGNED;
    if (io->inst_masks && !io->inst_bits) return BT_ERR_BAD_ARG;   // the bytes are expanded from the bits
    if ((io->inst_bits && !aligned16(io->inst_bits)) || (io->inst_masks && !aligned16(io->inst_masks))) return BT_ERR_MISALIGNED;
    if (io->seg_sweep && (!io->seg_img3 || !io->seg_prob_sum)) return BT_ERR_BAD_ARG;   // the record's IoU and score inputs
    if (io->seg_sweep && !aligned16(io->seg_sweep)) return BT_ERR_MISALIGNED;
    if (const BtIOSoftDice *sd = soft_io(*p, *io))
        if ((sd->seg_soft_dice || sd->seg_soft_acc) && !sd->seg_soft2) return BT_ERR_BAD_ARG;   // computed from its sums
    return BT_OK;
}

// Helper streams of btpost_run: the GT-bit packing (independent of the detections) runs beside the decode / NMS
// kernels, which leave most SMs idle, and the COCO matching beside the mask kernels.  A helper stream is forked from
// and joined back into the caller's stream with events, so the whole call is still ordered on the caller's stream and
// capturable into a CUDA graph.  Every call borrows a (stream, 5 events) set from a per-device pool under a mutex and
// returns it when its launches are enqueued: concurrent calls from several host threads get distinct sets (re-entrant),
// consecutive calls reuse one (a cudaStreamWaitEvent refers to the record that precedes it, so re-recording an
// event afterwards is harmless).  Host-side objects only; no device memory.
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, pack = nullptr, nms = nullptr, gather = nullptr, join = nullptr;
    SideStream *next = nullptr;
};
static std::mutex g_side_mutex;
static SideStream *g_side_free[64] = {};
static SideStream *side_acquire(int *dev_out) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    *dev_out = dev;
    {
        std::lock_guard<std::mutex> lk(g_side_mutex);
        if (SideStream *t = g_side_free[dev]) { g_side_free[dev] = t->next; t->next = nullptr; return t; }
    }
    SideStream *t = new (std::nothrow) SideStream();
    if (!t) return nullptr;
    bool ok = cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking) == cudaSuccess;
    cudaEvent_t *ev[5] = {&t->fork, &t->pack, &t->nms, &t->gather, &t->join};
    for (auto e : ev) ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {   // do not pool a half-built set
        for (auto e : ev) if (*e) cudaEventDestroy(*e);
        if (t->stream) cudaStreamDestroy(t->stream);
        delete t;
        return nullptr;
    }
    return t;
}
static void side_release(SideStream *t, int dev) {
    std::lock_guard<std::mutex> lk(g_side_mutex);
    t->next = g_side_free[dev];
    g_side_free[dev] = t;
}

#ifdef BT_DEBUG_HOOKS
int g_debug_skip = 0;   // developer tool (scripts/ablate.py, debug build only): launches left out of btpost_run
#endif

}  // namespace bt

using namespace bt;

extern "C" {

#ifdef BT_DEBUG_HOOKS
// Developer tool of the debug build (libbtpost_dbg.so, `make dbg`); the product library does not contain it.  Leaves
// kernels out of the following btpost_run calls to measure what each costs with several batches in flight (results
// are then stale / invalid).
// bits: 1 gt_pack, 2 decode_filter, 4 nms, 8 plan, 16 gather, 32 match, 64 contract, 128 cells + finalize
BTPOST_API int btpost_debug_skip(int mask) { bt::g_debug_skip = mask; return BT_OK; }
#endif

int btpost_version(void) { return BTPOST_VERSION; }

const char *btpost_error_string(int code) {
    switch (code) {
        case BT_OK: return "ok";
        case BT_ERR_BAD_ARG: return "bad argument (null pointer, non-positive size or inconsistent parameters)";
        case BT_ERR_UNSUPPORTED: return "unsupported shape (need nm=32, proto=img/4, img_w%32==0, nc<=16, max_gt<=32, max_det<=4096, and at most 32768 "
                                         "anchors; an L2 head with N % 4 != 0 at most 8192)";
        case BT_ERR_WORKSPACE: return "workspace too small (see btpost_workspace_bytes)";
        case BT_ERR_MISALIGNED: return "misaligned pointer (workspace 256 B; head/protos/masks 16 B)";
        case BT_ERR_CUDA: return "CUDA launch failed";
        case BT_ERR_NCCL: return "NCCL call failed";
        default: return "unknown error";
    }
}

int btpost_workspace_bytes(const BtParams *p, size_t *bytes) {
    if (!p || !bytes) return BT_ERR_BAD_ARG;
    if (p->batch <= 0 || p->num_anchors <= 0) return BT_ERR_BAD_ARG;
    if (int rc = check_anchor_limit(p)) return rc;   // a configuration btpost_run would reject fails here already
    *bytes = carve(p, nullptr).bytes;
    return BT_OK;
}

int btpost_decode_filter(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream) {
    int rc = check_params(p, io);
    if (rc == BT_OK) rc = check_ws(p, ws, ws_bytes);
    if (rc == BT_OK) rc = check_stage1(p, io);
    if (rc != BT_OK) return rc;
    return launch_decode_filter(*p, *io, carve(p, ws), static_cast<cudaStream_t>(stream));
}

int btpost_nms_match(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream) {
    int rc = check_params(p, io);
    if (rc == BT_OK) rc = check_ws(p, ws, ws_bytes);
    if (rc == BT_OK) rc = check_stage2(p, io);
    if (rc != BT_OK) return rc;
    return launch_nms_match(*p, *io, carve(p, ws), static_cast<cudaStream_t>(stream));
}

int btpost_masks(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream) {
    return btpost_masks_parts(p, io, ws, ws_bytes, stream, BT_MASKS_PACK | BT_MASKS_CONTRACT | BT_MASKS_CELLS);
}

int btpost_masks_parts(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream, int parts) {
    int rc = check_params(p, io);
    if (rc == BT_OK) rc = check_ws(p, ws, ws_bytes);
    if (rc == BT_OK) rc = check_stage3(p, io);
    if (rc == BT_OK && (parts & ~7)) rc = BT_ERR_BAD_ARG;
    if (rc != BT_OK) return rc;
    return launch_masks(*p, *io, carve(p, ws), static_cast<cudaStream_t>(stream), parts);
}

int btpost_run(const BtParams *p, const BtIO *io, void *ws, size_t ws_bytes, void *stream) {
    int rc = check_params(p, io);
    if (rc == BT_OK) rc = check_ws(p, ws, ws_bytes);
    if (rc == BT_OK) rc = check_stage1(p, io);
    if (rc == BT_OK) rc = check_stage2(p, io);
    if (rc == BT_OK) rc = check_stage3(p, io);
    if (rc != BT_OK) return rc;
    Workspace w = carve(p, ws);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int dev = 0;
    SideStream *side = side_acquire(&dev);
    if (!side) return BT_ERR_CUDA;
    auto ok = [](cudaError_t e) { return e == cudaSuccess; };
#ifdef BT_DEBUG_HOOKS
    const int skip = g_debug_skip;
#else
    constexpr int skip = 0;
#endif
    // fork: GT bits on the helper stream while the caller's stream decodes, filters and runs the NMS
    if (!ok(cudaEventRecord(side->fork, s)) || !ok(cudaStreamWaitEvent(side->stream, side->fork, 0))) {
        side_release(side, dev);
        return BT_ERR_CUDA;   // nothing was enqueued on the helper stream yet
    }
    if (!(skip & 1)) rc = launch_masks(*p, *io, w, side->stream, BT_MASKS_PACK);
    else cudaMemsetAsync(w.work, 0, 32 * 32 * sizeof(int32_t), side->stream);   // ablation: the queue counters gt_pack resets
    if (rc == BT_OK && !ok(cudaEventRecord(side->pack, side->stream))) rc = BT_ERR_CUDA;
    if (rc == BT_OK && !(skip & 2)) rc = launch_decode_filter(*p, *io, w, s);
    // NMS, then the mask-stage plan on the caller's stream while the helper stream gathers the kept detections' mask
    // coefficients and runs the COCO matching (beside the mask kernels)
    if (rc == BT_OK && !(skip & 4)) rc = launch_nms_match(*p, *io, w, s, BT_NMS_SORT_SWEEP);
    else if (rc == BT_OK) {   // ablation: the counters the NMS kernel resets for the plan
        cudaMemsetAsync(w.pool_used, 0, sizeof(unsigned long long), s);
        cudaMemsetAsync(w.n_items, 0, 2 * sizeof(int32_t), s);
    }
    if (rc == BT_OK && (!ok(cudaEventRecord(side->nms, s)) || !ok(cudaStreamWaitEvent(side->stream, side->nms, 0)))) rc = BT_ERR_CUDA;
    if (rc == BT_OK && !(skip & 8)) rc = launch_nms_match(*p, *io, w, s, BT_NMS_PLAN);
    if (rc == BT_OK && !(skip & 16)) rc = launch_nms_match(*p, *io, w, side->stream, BT_NMS_GATHER);
    if (rc == BT_OK && !ok(cudaEventRecord(side->gather, side->stream))) rc = BT_ERR_CUDA;
    if (rc == BT_OK && !(skip & 32)) rc = launch_nms_match(*p, *io, w, side->stream, BT_NMS_COCO);
    // join point of the helper stream: recorded whatever happened above (after the last launch attempt on it), so that
    // the wait below never refers to a stale record of an earlier call and a capture never ends with an unjoined stream
    const bool join_rec = ok(cudaEventRecord(side->join, side->stream));
    if (rc == BT_OK && !join_rec) rc = BT_ERR_CUDA;
    if (rc == BT_OK && (!ok(cudaStreamWaitEvent(s, side->pack, 0)) || !ok(cudaStreamWaitEvent(s, side->gather, 0)))) rc = BT_ERR_CUDA;
    if (rc == BT_OK && (skip & (64 | 128)) != (64 | 128))
        rc = launch_masks(*p, *io, w, s, ((skip & 64) ? 0 : BT_MASKS_CONTRACT) | ((skip & 128) ? 0 : BT_MASKS_CELLS));
    if (join_rec && !ok(cudaStreamWaitEvent(s, side->join, 0)) && rc == BT_OK) rc = BT_ERR_CUDA;
    side_release(side, dev);
    return rc;
}

int btpost_seg_curve(const BtParams *p, void *ws, size_t ws_bytes, const float *thresholds, int32_t num_thresholds,
                     int64_t *hist, void *stream) {
    if (!thresholds || !hist) return BT_ERR_BAD_ARG;
    if (num_thresholds < 2 || num_thresholds > BT_MAX_CURVE_THRS) return BT_ERR_BAD_ARG;
    for (int i = 0; i < num_thresholds; ++i) {
        const float v = thresholds[i];
        if (!(v >= 0.0f && v <= 1.0f)) return BT_ERR_BAD_ARG;   // NaN fails too
        if (i > 0 && v < thresholds[i - 1]) return BT_ERR_BAD_ARG;
    }
    if (reinterpret_cast<uintptr_t>(hist) & 7) return BT_ERR_MISALIGNED;
    int rc = check_shape(p);
    if (rc == BT_OK) rc = check_ws(p, ws, ws_bytes);
    if (rc != BT_OK) return rc;
    return launch_seg_curve(*p, carve(p, ws), thresholds, num_thresholds, hist, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
