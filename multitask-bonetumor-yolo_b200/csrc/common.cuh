// Shared device/host helpers of libbtpost (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/btpost.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libbtpost is written for sm_100a (B200) only"
#endif

// Optional per-phase cycle accounting (debug builds only: make dbg).  Thread 0 of every CTA adds the
// cycles it spent between marks into a global table read back by btpost_debug_phase_cycles().
#ifdef BT_PHASE_TIMING
// (defined in nms_match.cu, the only file with marks: no relocatable device code needed)
#define BT_PHASE_INIT() long long _pt = clock64()
#define BT_PHASE_MARK(kern, idx)                                                           \
    do {                                                                                   \
        if (threadIdx.x == 0) {                                                            \
            long long _n = clock64();                                                      \
            atomicAdd(&g_phase_cycles[kern][idx], (unsigned long long)(_n - _pt));         \
            _pt = _n;                                                                      \
        }                                                                                  \
    } while (0)
#else
#define BT_PHASE_INIT() do {} while (0)
#define BT_PHASE_MARK(kern, idx) do {} while (0)
#endif

namespace bt {

// sigmoid(x) > 0.5 in fp32 (src/running_main_v2.py:702-703, src/test_model.py:85) holds exactly
// for x > 1.5 * 2^-24 (pinned against torch in tests/golden/make_golden.py).
__device__ __forceinline__ bool sigmoid_gt_half(float x) { return x > 8.940696716308594e-08f; }

// exp shared bit-for-bit with oracle/btpost_oracle.c::bto_expf (Cody-Waite + degree-6 polynomial,
// fma/mul/add only).  No overflow guard: the exponent add wraps above x ~ 88.
__device__ __forceinline__ float bt_expf(float x) {
    if (x < -87.0f) return 0.0f;
    float t = __fmul_rn(x, 1.4426950408889634f);
    float n = rintf(t);
    float r = __fmaf_rn(n, -0.693145751953125f, x);
    r = __fmaf_rn(n, -1.428606765330187e-06f, r);
    float p = 1.3888889225e-03f;
    p = __fmaf_rn(p, r, 8.3333337680e-03f);
    p = __fmaf_rn(p, r, 4.1666667908e-02f);
    p = __fmaf_rn(p, r, 1.6666667163e-01f);
    p = __fmaf_rn(p, r, 0.5f);
    p = __fmaf_rn(p, r, 1.0f);
    p = __fmaf_rn(p, r, 1.0f);
    int e = (int)n;
    return __int_as_float(__float_as_int(p) + (e << 23));
}

// sigmoid(x) in units of 2^-40, the term of the soft-Dice sums (BtIOSoftDice.seg_soft2): 1 / (1 + bt_expf(-x)) rounded once
// per operation, then scaled (exactly) and rounded to the nearest integer.  x < -87 gives 0: bt_expf(-x) would
// wrap there, and the true value is below 2^-125, which rounds to 0 in this fixed point anyway.
__device__ __forceinline__ long long soft_prob_fx40(float x) {
    if (x < -87.0f) return 0ll;
    const float p = __fdiv_rn(1.0f, __fadd_rn(1.0f, bt_expf(-x)));
    return __float2ll_rn(__fmul_rn(p, 1099511627776.0f));
}

// Order-preserving image of an fp32 score: ascending key = descending score (sort keys of the NMS, sweep records).
__device__ __forceinline__ uint32_t desc_key(float s) {
    uint32_t u = __float_as_uint(s);
    if (s != s) return 0u;                                   // NaN sorts first
    if (u == 0x80000000u) u = 0u;                            // -0.0 == +0.0
    uint32_t asc = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return ~asc;                                             // smaller key = higher score
}

// COCOeval area ranges (all, small, medium, large), bounds inclusive: an area lies outside range a when it is below
// COCO_AREA_LO[a] or above COCO_AREA_HI[a].  Brace initialisers of a kernel's local const arrays.
#define COCO_AREA_LO {0.0, 0.0, 32.0 * 32.0, 96.0 * 96.0}
#define COCO_AREA_HI {1e10, 32.0 * 32.0, 96.0 * 96.0, 1e10}

// Crop region of a detection at prototype resolution: pixels with r>=y1 & r<y2 & c>=x1 & c<x2
// on the box scaled by proto/img (Ultralytics crop_mask).  Returns false for an empty region.
__device__ __forceinline__ bool crop_region(const float *o, int crop, float rx, float ry, int PW, int PH, int &r_lo,
                                            int &r_hi, int &c_lo, int &c_hi) {
    r_lo = 0; r_hi = PH - 1; c_lo = 0; c_hi = PW - 1;
    if (!crop) return true;
    float x1 = __fmul_rn(o[0], rx), y1 = __fmul_rn(o[1], ry), x2 = __fmul_rn(o[2], rx), y2 = __fmul_rn(o[3], ry);
    if (!((x1 == x1) && (y1 == y1) && (x2 == x2) && (y2 == y2))) return false;
    c_lo = max(0, (int)ceilf(fmaxf(x1, -1.0f)));
    r_lo = max(0, (int)ceilf(fmaxf(y1, -1.0f)));
    c_hi = min(PW - 1, (int)ceilf(fminf(x2, (float)PW + 1.0f)) - 1);
    r_hi = min(PH - 1, (int)ceilf(fminf(y2, (float)PH + 1.0f)) - 1);
    return c_lo <= c_hi && r_lo <= r_hi;
}

// Workspace carve-up (all offsets 256-byte aligned).
struct Workspace {
    float4 *cand_box;     // [B, cap]
    float *cand_score;    // [B, cap]
    int32_t *cand_label;  // [B, cap]
    int32_t *cand_anchor; // [B, cap]
    unsigned long long *sort_keys;  // [B, sort_stride_u64(cap)] (lists that do not fit the shared-memory sorts)
    int32_t *acc;         // [B, 8] per-image int counters: seg inter,P,G ; uni inter,P,G
    short4 *det_region;   // [B, K] crop region of each kept detection at prototype resolution (r_lo, r_hi, c_lo, c_hi)
    int32_t *scr_off;     // [B, K] offset (floats) of the detection's crop-box logits in `pool`; -1: none (invalid / pool full)
    unsigned long long *pool_used;   // [1] floats handed out of `pool` in this call
    int32_t *work;        // [32 * 32] work-queue counters of cells_kernel (one per 128 bytes)
    int32_t *gpart;       // [B, NBY] GT pixels per row of cell blocks
    unsigned long long *gtc, *unc;   // [B, NBY, NBX] GT / union-of-instance-masks bits per 2x2 block of cells
    float *lm;            // [B, PH, PW] projector logits at prototype resolution
    int32_t *tile_cnt;    // [B, tiles] detections listed on each contract_kernel tile
    unsigned short *tile_list;   // [B, tiles, K]
    int2 *items;          // [item_cap] work items of cells_kernel: (image * K + detection, chunk of C_CHUNK blocks)
    int32_t *n_items;     // [2]: number of items; [1] = 1 when some detection found no room in the pool
    long long item_cap;
    float *pool;          // [pool_cap] logits of the detections' crop boxes, back to back
    long long pool_cap;
    size_t bytes;
};

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// The soft-Dice outputs when the caller passed a BtIOSoftDice (BtParams.io_soft_dice), else null.  `io` is then its
// first member, so the cast recovers the enclosing struct.
static inline const BtIOSoftDice *soft_io(const BtParams &p, const BtIO &io) {
    return p.io_soft_dice ? reinterpret_cast<const BtIOSoftDice *>(&io) : nullptr;
}

// The candidate list holds every anchor that passes the filter (anchor order); BtParams.max_cand (Ultralytics max_nms)
// limits how many of them, best score first, enter the NMS sweep.
static inline int cand_capacity(const BtParams *p) { return p->num_anchors; }
static inline int cand_limit(const BtParams *p) {
    return (p->max_cand > 0 && p->max_cand < p->num_anchors) ? p->max_cand : p->num_anchors;
}


// 2x2 blocks of cells per dimension: cells -1 .. n-1 (a cell = the 4x4 output pixels between four prototype pixels)
static inline int mask_blocks(int n) { return (n + 2) / 2; }

// Logit pool of the mask stage: room for 16 full-image crop boxes per image (the synthetic workload uses ~2),
// shared by the batch; detections that do not fit are contracted corner by corner in cells_kernel.
static inline long long mask_pool_floats(const BtParams *p) {
    long long v = (long long)p->batch * 16 * p->proto_h * p->proto_w;
    const long long full = (long long)p->batch * p->max_det * p->proto_h * p->proto_w;
    if (v > full) v = full;
    return v > 0x7fffff00ll ? 0x7fffff00ll : v;
}

// contract_kernel tile (prototype pixels); the plan bins every detection into the tiles its crop box touches
constexpr int TA_W = 32, TA_H = 8;
constexpr int PLAN_MAX_TILES = 4096;
static inline int mask_tiles(const BtParams *p) { return ((p->proto_w + TA_W - 1) / TA_W) * ((p->proto_h + TA_H - 1) / TA_H); }

// cells_kernel works on chunks of C_CHUNK 2x2 cell blocks of one detection's crop box
constexpr int C_CHUNK = 128;
static inline long long mask_item_cap(const BtParams *p) {
    const long long per_det = ((long long)mask_blocks(p->proto_h) * mask_blocks(p->proto_w) + C_CHUNK - 1) / C_CHUNK;
    const long long v = (long long)p->batch * p->max_det * per_det;
    return v > 0x7fffff00ll ? 0x7fffff00ll : v;
}

static inline int next_pow2(int v) {
    int r = 1;
    while (r < v) r <<= 1;
    return r;
}

// Per-image slice of Workspace.sort_keys in 8-byte words: the bitonic network's padded key array, or the bucket sort's
// (key, index) pairs + 32-bit index list of a long candidate list (12 bytes per candidate, rounded up to 32 candidates).
static inline size_t sort_stride_u64(size_t cap) {
    const size_t pow2 = (size_t)next_pow2((int)cap), pairs = (cap + 31) / 32 * 32;
    const size_t bucket = pairs + (pairs + 1) / 2;
    return pow2 > bucket ? pow2 : bucket;
}

// Sorted candidates are consumed by the NMS kernel in shared-memory windows of this many.
constexpr int K2_TAIL_WIN = 1024;

static inline Workspace carve(const BtParams *p, void *base) {
    Workspace w;
    char *ptr = static_cast<char *>(base);
    size_t off = 0;
    const size_t B = (size_t)p->batch, cap = (size_t)cand_capacity(p);
    auto take = [&](size_t n) {
        char *r = ptr ? ptr + off : nullptr;
        off += align_up(n, 256);
        return r;
    };
    w.cand_box = reinterpret_cast<float4 *>(take(B * cap * sizeof(float4)));
    w.cand_score = reinterpret_cast<float *>(take(B * cap * sizeof(float)));
    w.cand_label = reinterpret_cast<int32_t *>(take(B * cap * sizeof(int32_t)));
    w.cand_anchor = reinterpret_cast<int32_t *>(take(B * cap * sizeof(int32_t)));
    w.sort_keys = reinterpret_cast<unsigned long long *>(take(B * sort_stride_u64(cap) * 8));
    w.acc = reinterpret_cast<int32_t *>(take(B * 8 * sizeof(int32_t)));
    w.det_region = reinterpret_cast<short4 *>(take(B * (size_t)p->max_det * sizeof(short4)));
    const size_t nby = (size_t)mask_blocks(p->proto_h), nbx = (size_t)mask_blocks(p->proto_w);
    w.scr_off = reinterpret_cast<int32_t *>(take(B * (size_t)p->max_det * sizeof(int32_t)));
    w.pool_used = reinterpret_cast<unsigned long long *>(take(sizeof(unsigned long long)));
    w.work = reinterpret_cast<int32_t *>(take(32 * 32 * sizeof(int32_t)));
    w.gpart = reinterpret_cast<int32_t *>(take(B * nby * sizeof(int32_t)));
    w.gtc = reinterpret_cast<unsigned long long *>(take(B * nby * nbx * 8));
    w.unc = reinterpret_cast<unsigned long long *>(take(B * nby * nbx * 8));
    w.lm = reinterpret_cast<float *>(take(B * (size_t)p->proto_h * p->proto_w * sizeof(float)));
    w.tile_cnt = reinterpret_cast<int32_t *>(take(B * (size_t)mask_tiles(p) * sizeof(int32_t)));
    w.tile_list = reinterpret_cast<unsigned short *>(take(B * (size_t)mask_tiles(p) * p->max_det * sizeof(unsigned short)));
    w.item_cap = mask_item_cap(p);
    w.items = reinterpret_cast<int2 *>(take((size_t)w.item_cap * sizeof(int2)));
    w.n_items = reinterpret_cast<int32_t *>(take(2 * sizeof(int32_t)));
    w.pool_cap = mask_pool_floats(p);
    w.pool = reinterpret_cast<float *>(take((size_t)w.pool_cap * sizeof(float)));
    w.bytes = off;
    return w;
}

int check_params(const BtParams *p, const BtIO *io);
int launch_decode_filter(const BtParams &p, const BtIO &io, const Workspace &w, cudaStream_t s);
// parts: BT_NMS_SORT_SWEEP (the NMS kernel) and, each needing only its results: BT_NMS_GATHER (mask coefficients of the
// kept detections), BT_NMS_PLAN (plan of the mask stage), BT_NMS_COCO (evaluateImg matching)
enum { BT_NMS_SORT_SWEEP = 1, BT_NMS_COCO = 2, BT_NMS_GATHER = 4, BT_NMS_PLAN = 8 };
int launch_nms_match(const BtParams &p, const BtIO &io, const Workspace &w, cudaStream_t s, int parts = 15);
// parts: BT_MASKS_PACK (GT bits; independent of the detections), BT_MASKS_CONTRACT (the pass over the prototypes),
// BT_MASKS_CELLS (upsample + threshold + counters + per-image finalize)
int launch_masks(const BtParams &p, const BtIO &io, const Workspace &w, cudaStream_t s, int parts = 7);

}  // namespace bt
