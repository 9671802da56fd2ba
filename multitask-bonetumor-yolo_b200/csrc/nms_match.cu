// Kernel group 2: per-image stable descending sort, greedy NMS with early exit at max_det, gather
// of the kept detections, COCOeval per-image matching.
//
// Reference statements replaced (paths under /root/reference/src):
//   NMS       running_main_v2.py:817  torchvision.ops.nms(item_boxes, item_top_scores, NMS_IOU)[:TOP_K]
//             (running_main_v3.py:549).  Keep indices are bit-exact: same ordering (stable
//             descending, NaN first, ties -> lower index), same fp32 IoU expression
//             inter / (area_i + area_j - inter) with one rounding per operation, same strict
//             comparison against the double threshold.
//   package   running_main_v2.py:818-839  ([K,4] boxes, [K] scores, [K] labels, [K,6] log rows)
//   matching  torchmetrics MeanAveragePrecision.update -> pycocotools COCOeval.evaluateImg
//             (configured at running_main_v2.py:228-251, evaluate_model.py:81-94; SURVEY.md A.3)
//
// B200 mapping.  nms_kernel, one CTA of 1024 / 512 / 256 threads per image:
//   1. sort    bucket rank sort (bucket_sort below): one pass -- min / max of the 32-bit descending
//              score keys, monotone map to 2048 buckets, histogram, scan, scatter of the 64-bit
//              (key, index) pairs, exact rank inside the bucket -- in shared memory, or in the
//              workspace for lists that do not fit.  Fallbacks for buckets of hundreds of equal
//              scores: stable LSD radix sort, 64-bit bitonic network with the keys in REGISTERS
//              (strides inside a thread are plain compare-exchanges, strides inside a warp are
//              shuffles, only the widest strides go through shared memory), the same network in
//              global memory.
//   2. sweep   the sorted list is staged in windows of 1024 and consumed 64 at a time:
//              (A) chunk vs KEPT boxes -- kept boxes are binned by the cell of their centre, and
//              for IoU thresholds >= 0.55 a suppressing pair has each centre inside the other
//              box, so a candidate only meets the kept boxes in the cells under its own box;
//              (B) "who suppresses me" rows among the candidates A left undecided (warp ballots;
//              the exact IoU only runs when some lane passes the cheap necessary condition);
//              (C) one warp resolves the chunk as a fixpoint over those rows.  Because keeps are
//              emitted in score order `[:TOP_K]` is an early exit, and because only KEPT or still
//              undecided boxes are ever tested against, a cluster of hundreds of candidates on one
//              object costs ~n tests, not n^2 (r01f: an all-pairs bit matrix, even spatially
//              culled, spent 365 k cycles per image there).
//   3. package boxes / scores / labels / keep indices / crop regions of the kept detections.
// The exact IoU decision uses a guarded approximate division (see suppresses()).
// coeff_gather_kernel spreads the mask-coefficient gather (K x 32 scattered 4-byte reads per image:
// latency-bound on one SM, r01e 16 us; gathering for every CANDIDATE in the decode kernel instead
// tripled the scattered DRAM sectors and cost 19 us, r01u) over the whole GPU.  match_kernel runs
// COCOeval's per-image matching, one CTA per image; the mask kernel is launched as its programmatic
// dependent and overlaps it.
#include <stdlib.h>

#ifdef BT_PHASE_TIMING
#include <cuda_runtime.h>
__device__ unsigned long long g_phase_cycles[3][16];
#endif
#include "common.cuh"

#ifdef BT_PHASE_TIMING
extern "C" __attribute__((visibility("default"))) int btpost_debug_phase_cycles(unsigned long long *out48, int reset) {
    if (cudaMemcpyFromSymbol(out48, g_phase_cycles, sizeof(unsigned long long) * 48) != cudaSuccess) return BT_ERR_CUDA;
    if (reset) {
        static unsigned long long zeros[48];
        if (cudaMemcpyToSymbol(g_phase_cycles, zeros, sizeof(zeros)) != cudaSuccess) return BT_ERR_CUDA;
    }
    return BT_OK;
}
#endif

namespace bt {

constexpr int NMS_CHUNK = 64;
constexpr int NMS_MINB_512 = 3;     // CTAs per SM the 512-thread variant is compiled for (3: 40 registers, measured in profiles/r02c_summary.md)
constexpr int NMS_WIN_512 = 1024;   // sorted candidates staged per window by the 512-thread variant
constexpr int A_SUBS_WIDE = 8;      // phase A threads per candidate of the 512- and 1024-thread variants
constexpr int SORT_REG_MAX = 16384;  // keys sorted in registers (16 per thread) up to this many
constexpr int SORT_SMALL_MAX = 4096; // same for the 512-thread variant (8 per thread): its shared memory stays below 80 KB
constexpr int GM_THREADS = 256;      // match_kernel block
constexpr int MAX_CELLS = 256;

// i = earlier (kept) box, j = later candidate; operand order of std::max/std::min as in
// torchvision's nms_kernel_impl so NaN coordinates behave identically.
//
// centre_cull: IoU > 0.5 means the intersection covers more than half of EACH box, hence contains
// each box's centre.  With iou_thres >= 0.55 (margin >> fp32 rounding of the IoU) a pair whose
// later centre (cxj, cyj) is outside the earlier box can be skipped without evaluating the IoU;
// every pair that is evaluated uses the exact expression, so the keep set does not change.
struct FastDiv { int on; float lo, hi; };
__device__ __forceinline__ bool suppresses(const float4 &bi, float ai, int li, const float4 &bj, float aj, int lj,
                                           float thr_up, int early_out, int class_mode, int centre_cull, float cxj,
                                           float cyj, const FastDiv &g_fast) {
    if (class_mode == BT_CLASS_AWARE && li != lj) return false;
    if (centre_cull && !(cxj >= bi.x && cxj <= bi.z && cyj >= bi.y && cyj <= bi.w)) return false;
    float xx1 = (bi.x < bj.x) ? bj.x : bi.x;
    float yy1 = (bi.y < bj.y) ? bj.y : bi.y;
    float xx2 = (bj.z < bi.z) ? bj.z : bi.z;
    float yy2 = (bj.w < bi.w) ? bj.w : bi.w;
    float w = __fsub_rn(xx2, xx1), h = __fsub_rn(yy2, yy1);
    w = (0.0f < w) ? w : 0.0f;
    h = (0.0f < h) ? h : 0.0f;
    float inter = __fmul_rn(w, h);
    if (early_out && !(inter > 0.0f)) return false;
    const float den = __fsub_rn(__fadd_rn(ai, aj), inter);
    // ovr = fl(inter / den) >= thr_up.  The approximate quotient (<= 2 ulp off for den < 2^126)
    // settles every pair that is not within 1e-6 (relative) of the threshold; only those pay for
    // the IEEE division, so the decision is the exact one for every input.
    if (g_fast.on && den < 1e37f && den > 1e-30f) {
        const float q = __fdividef(inter, den);
        if (q > g_fast.hi) return true;
        if (q < g_fast.lo) return false;
    }
    return __fdiv_rn(inter, den) >= thr_up;
}

__device__ __forceinline__ float box_area(const float4 &b) { return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y)); }

__device__ __forceinline__ double bb_iou(const double *d, const double *g) {
    double w = fmin(d[0] + d[2], g[0] + g[2]) - fmax(d[0], g[0]);
    if (w <= 0) return 0.0;
    double h = fmin(d[1] + d[3], g[1] + g[3]) - fmax(d[1], g[1]);
    if (h <= 0) return 0.0;
    double i = w * h;
    return i / (d[2] * d[3] + g[2] * g[3] - i);
}


struct K2Params {
    int N, nc, nm, C, cap, cap_pow2, limit, max_det, max_gt, class_mode, layout;   // limit: BtParams.max_cand (best-scoring candidates that enter the sweep)
    float thr_up;     // smallest float f with (double)f > iou_thres:  (double)ovr > thr  <=>  ovr >= thr_up
    FastDiv fast;     // guarded approximate division (see suppresses)
    int early_out;    // iou_thres >= 0: pairs with zero intersection can never be suppressed
    float max_wh;
    const void *head;     // L2: coefficients are rows 4+nc.. of the head (fp32 or bf16)
    int head_bf16;
    const void *coeffs;   // L1: [B, nm, N] (fp32, or bf16 with the maps)
    const float4 *cand_box;
    const float *cand_score;
    const int32_t *cand_label, *cand_anchor, *n_cand;
    unsigned long long *sort_keys;
    int32_t *det_count;
    float *dets;
    int64_t *det_keep;
    int32_t *det_anchor;
    float *det_coeff;
    // GT + COCO
    const int32_t *gt_count;
    const float *gt_boxes;
    const int32_t *gt_labels;
    int T;
    double thrs[BT_MAX_IOU_THRS];
    int32_t *dt_match;
    uint8_t *dt_ignore, *gt_ignore;
    // accumulators of the mask kernel, zeroed here
    int32_t *acc, *inst_area, *inst_inter;
    double *seg_prob_sum;
    int region0_bytes;    // shared region 0: list of candidate indices in NMS order
    size_t sort_stride;   // u64 words per image of sort_keys
    int bucket_max;       // longest list the bucket rank sort takes (shared memory behind region 0 holds its pairs)
    int crop, PW, PH; float rx, ry; short4 *det_region;   // crop regions for the mask kernel
    int32_t *scr_off; unsigned long long *pool_used; long long pool_cap;   // logit-pool plan of the mask stage
    int2 *items; int32_t *n_items; int item_cap;                            // work items of cells_kernel
    int32_t *tile_cnt; unsigned short *tile_list; int ntiles, ntx;         // tile lists of contract_kernel
    int centre_cull; // iou_thres >= 0.55: a suppressing pair has each centre inside the other box
    int gx, gy; float inv_cw, inv_ch;   // centre-cell grid
    int coco_smem_doubles;
    long long *sweep;     // optional sweep state (header + record ring, include/btpost.h)
    int image_offset, drop_gt_no_cand;
    const int32_t *image_base;
    long long *seg_soft2;   // soft-Dice sums of the mask kernel (optional), zeroed here; last: earlier offsets stay
};

// =================================================================================================
// sort
// =================================================================================================
__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m) {
    unsigned lo = __shfl_xor_sync(0xffffffffu, (unsigned)v, m), hi = __shfl_xor_sync(0xffffffffu, (unsigned)(v >> 32), m);
    return ((unsigned long long)hi << 32) | lo;
}

// Bitonic sort (ascending) of P2 = nthr * E keys; thread t < nthr holds elements t*E .. t*E+E-1.
// Every thread of the block must call this (block barriers in the shared-memory steps).
template <int E>
__device__ __forceinline__ void bitonic_regs(unsigned long long (&v)[E], unsigned long long *s_x, int tid, int nthr) {
    const bool active = tid < nthr;
    const int P2 = nthr * E;
    for (int k = 2; k <= P2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32 * E) {
                if (active) {
#pragma unroll
                    for (int e = 0; e < E; ++e) s_x[tid * E + e] = v[e];
                }
                __syncthreads();
                if (active) {
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        const int i = tid * E + e;
                        const unsigned long long o = s_x[i ^ j];
                        const bool keep_min = ((i & j) == 0) == ((i & k) == 0);
                        v[e] = ((o < v[e]) == keep_min) ? o : v[e];
                    }
                }
                __syncthreads();
            } else if (j >= E) {
                if (active) {
                    const int tj = j / E;
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        const int i = tid * E + e;
                        const unsigned long long o = shfl_xor_u64(v[e], tj);
                        const bool keep_min = ((tid & tj) == 0) == ((i & k) == 0);
                        v[e] = ((o < v[e]) == keep_min) ? o : v[e];
                    }
                }
            } else if (active) {
#pragma unroll
                for (int jj = E >> 1; jj >= 1; jj >>= 1) {
                    if (jj != j) continue;
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        if (e & jj) continue;
                        const int i = tid * E + e;
                        const bool asc = (i & k) == 0;
                        const unsigned long long a = v[e], c = v[e | jj];
                        if ((a > c) == asc) { v[e] = c; v[e | jj] = a; }
                    }
                }
            }
        }
    }
}

// Sorts the image's candidates; on return s_sidx[i] (i < M) = index of the i-th candidate in NMS order.
template <int E>
__device__ __forceinline__ void sort_to_smem(const float *cscore, int M, int nthr, unsigned long long *s_x, uint32_t *s_sidx) {
    const int tid = threadIdx.x;
    unsigned long long v[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int i = tid * E + e;
        v[e] = (tid < nthr && i < M) ? (((unsigned long long)desc_key(__ldg(cscore + i)) << 32) | (unsigned)i) : ~0ull;
    }
    bitonic_regs<E>(v, s_x, tid, nthr);
    __syncthreads();   // s_x (aliases s_sidx) is no longer read
    if (tid < nthr) {
#pragma unroll
        for (int e = 0; e < E; ++e) s_sidx[tid * E + e] = (uint32_t)v[e];
    }
    __syncthreads();
}

// Stable LSD radix sort (four passes of 8 bits) of the 32-bit descending score keys for lists of <= RADIX_MAX
// candidates: stability gives "ties -> lower index" for free, so only 32-bit keys are compared, and a pass is two
// walks of 32 candidates per warp step (match.any on the digit) plus one block scan -- a fifth of the instructions of
// the 64-bit bitonic network and a third of its barriers.  Warp w owns a contiguous tile of the list; counters are
// laid out digit-major ([256][warps]) so their exclusive scan is the stable order.  On return s_sidx[i] (i < M) =
// index of the i-th candidate in NMS order.  Every thread of the block must call this.
constexpr int RADIX_MAX = 2048;
// lanes of the warp that hold the same digit: 8 independent ballots
__device__ __forceinline__ unsigned digit_peers(int d, bool valid) {
    unsigned peers = __ballot_sync(0xffffffffu, valid);
#pragma unroll
    for (int bit = 0; bit < 8; ++bit) {
        const bool one = (d >> bit) & 1;
        const unsigned bm = __ballot_sync(0xffffffffu, one);
        peers &= one ? bm : ~bm;
    }
    return peers;
}
template <int NT>
__device__ __forceinline__ void radix_sort_to_smem(const float *cscore, int M, unsigned char *smem_raw, uint32_t *s_sidx) {
    constexpr int NW = NT / 32;
    __shared__ int s_wsum[32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int Mp = (M + 31) & ~31;
    unsigned long long *bufA = reinterpret_cast<unsigned long long *>(smem_raw), *bufB = bufA + Mp;
    uint32_t *hist = reinterpret_cast<uint32_t *>(bufB + Mp);   // [256 * NW]
    const int nchunks = Mp >> 5, cpw = (nchunks + NW - 1) / NW;
    const int c_lo = min(wid * cpw, nchunks), c_hi = min(c_lo + cpw, nchunks);
    const unsigned lt = (1u << lane) - 1u;
    for (int i = tid; i < M; i += NT) bufA[i] = ((unsigned long long)desc_key(__ldg(cscore + i)) << 32) | (unsigned)i;
#pragma unroll 1
    for (int pass = 0; pass < 4; ++pass) {
        const unsigned long long *src = (pass & 1) ? bufB : bufA;
        unsigned long long *dst = (pass & 1) ? bufA : bufB;
        const int shift = 32 + 8 * pass;
        for (int i = tid; i < 256 * NW; i += NT) hist[i] = 0;
        __syncthreads();
        for (int c = c_lo; c < c_hi; ++c) {
            const int i = c * 32 + lane;
            const bool valid = i < M;
            const int d = valid ? (int)((src[valid ? i : 0] >> shift) & 255ull) : 256;
            const unsigned peers = digit_peers(d, valid);
            if (valid && lane == __ffs(peers) - 1) hist[d * NW + wid] += __popc(peers);
            __syncwarp();
        }
        __syncthreads();
        {   // exclusive scan of the 256 * NW counters: 8 consecutive ones per thread
            uint4 *h4 = reinterpret_cast<uint4 *>(hist) + 2 * tid;
            uint4 a = h4[0], b = h4[1];
            const unsigned v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
            unsigned ex[8], sum = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { ex[j] = sum; sum += v[j]; }
            unsigned incl = sum;
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) {
                const unsigned u = __shfl_up_sync(0xffffffffu, incl, dd);
                if (lane >= dd) incl += u;
            }
            if (lane == 31) s_wsum[wid] = (int)incl;
            __syncthreads();
            const unsigned wv = lane < NW ? (unsigned)s_wsum[lane] : 0u;
            unsigned winc = wv;
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) {
                const unsigned u = __shfl_up_sync(0xffffffffu, winc, dd);
                if (lane >= dd) winc += u;
            }
            const unsigned base = __shfl_sync(0xffffffffu, winc - wv, wid) + incl - sum;
            a = make_uint4(ex[0] + base, ex[1] + base, ex[2] + base, ex[3] + base);
            b = make_uint4(ex[4] + base, ex[5] + base, ex[6] + base, ex[7] + base);
            h4[0] = a; h4[1] = b;
        }
        __syncthreads();
        for (int c = c_lo; c < c_hi; ++c) {
            const int i = c * 32 + lane;
            const bool valid = i < M;
            const unsigned long long e = src[valid ? i : 0];
            const int d = valid ? (int)((e >> shift) & 255ull) : 256;
            const unsigned peers = digit_peers(d, valid);
            unsigned rank = 0;
            if (valid) rank = hist[d * NW + wid] + __popc(peers & lt);
            __syncwarp();
            if (valid && lane == __ffs(peers) - 1) hist[d * NW + wid] += __popc(peers);
            __syncwarp();
            if (valid) {
                if (pass < 3) dst[rank] = e;
                else s_sidx[rank] = (uint32_t)e;   // the keys are not needed any more: the index list lands where bufA was
            }
        }
        __syncthreads();
    }
}

// Bucket rank sort (lists of <= P.bucket_max candidates; the default path).  The four radix passes above cost 31 k cycles
// per image at ~930 candidates (r02c phase counters: a third of the kernel) in barriers and dependent shuffle chains;
// this is one pass: (1) min / max of the 32-bit descending keys, (2) a MONOTONE map key -> one of BUCKETS buckets
// (float scale of key - min: conversion, product and truncation are all non-decreasing, equal keys share a bucket),
// histogram with shared-memory atomics, (3) exclusive scan of the counters, (4) scatter of the 64-bit (key, index)
// pairs into their bucket's range in any order, (5) every element counts the pairs of its own bucket that compare
// below it: bucket start + that count is its exact rank in the (key, index) order, i.e. the stable order
// ("ties -> lower index").  The result does not depend on the bucket map or on the order of the atomics.  A list
// with a bucket of more than BUCKET_OCC_MAX entries (hundreds of equal scores) returns false without having written
// s_sidx and the caller takes the radix / bitonic path.  Every thread of the block must call this.
// Lists that fit (<= P.bucket_max): the index list is [0, 4 M) of shared region 0, pairs and counters overlay the window
// area behind it.  Longer lists (GLOBAL): pairs and the index list live in the image's slice of the workspace sort
// buffer, only the counters are in shared memory -- one pass over the L2 instead of the ~100 barrier-separated stages
// of a bitonic network in global memory.
constexpr int BUCKETS = 2048;
constexpr int BUCKET_OCC_MAX = 256;
template <int NT, bool GLOBAL>
__device__ __forceinline__ bool bucket_sort(const float *cscore, int M, unsigned long long *buf, int *start, uint32_t *out) {
    constexpr int NW = NT / 32, PER = BUCKETS / NT;
    __shared__ unsigned s_kmin, s_kmax, s_occ;
    __shared__ int s_bsum[32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    int *cur = start + BUCKETS;                                                                     // [BUCKETS]
    if (tid == 0) { s_kmin = 0xffffffffu; s_kmax = 0u; s_occ = 0u; }
#pragma unroll
    for (int j = 0; j < PER; ++j) start[tid * PER + j] = 0;
    __syncthreads();
    {
        unsigned lo = 0xffffffffu, hi = 0u;
        for (int i = tid; i < M; i += NT) {
            const unsigned k = desc_key(__ldg(cscore + i));
            lo = min(lo, k); hi = max(hi, k);
        }
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        if (lane == 0) { atomicMin(&s_kmin, lo); atomicMax(&s_kmax, hi); }
    }
    __syncthreads();
    const unsigned kmin = s_kmin;
    const float scale = __fdiv_rn((float)BUCKETS, __fadd_rn(__uint2float_rn(s_kmax - kmin), 1.0f));
    auto bucket_of = [&](unsigned k) { return min(__float2int_rz(__fmul_rn(__uint2float_rn(k - kmin), scale)), BUCKETS - 1); };
    for (int i = tid; i < M; i += NT) atomicAdd(&start[bucket_of(desc_key(__ldg(cscore + i)))], 1);
    __syncthreads();
    {   // exclusive scan of the counters, PER consecutive ones per thread
        int v[PER], sum = 0, occ = 0;
#pragma unroll
        for (int j = 0; j < PER; ++j) { v[j] = start[tid * PER + j]; occ = max(occ, v[j]); sum += v[j]; }
        int incl = sum;
#pragma unroll
        for (int dd = 1; dd < 32; dd <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, incl, dd);
            if (lane >= dd) incl += u;
        }
        occ = __reduce_max_sync(0xffffffffu, occ);
        if (lane == 31) s_bsum[wid] = incl;
        if (lane == 0 && occ > BUCKET_OCC_MAX) atomicMax(&s_occ, (unsigned)occ);
        __syncthreads();
        const int wv = lane < NW ? s_bsum[lane] : 0;
        int winc = wv;
#pragma unroll
        for (int dd = 1; dd < 32; dd <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, winc, dd);
            if (lane >= dd) winc += u;
        }
        int run = __shfl_sync(0xffffffffu, winc - wv, wid) + incl - sum;
#pragma unroll
        for (int j = 0; j < PER; ++j) { start[tid * PER + j] = run; cur[tid * PER + j] = run; run += v[j]; }
    }
    __syncthreads();
    if (s_occ) return false;   // block-uniform
    for (int i = tid; i < M; i += NT) {
        const unsigned k = desc_key(__ldg(cscore + i));
        buf[atomicAdd(&cur[bucket_of(k)], 1)] = ((unsigned long long)k << 32) | (unsigned)i;
    }
    __syncthreads();
    for (int p = tid; p < M; p += NT) {
        // GLOBAL: the pairs were written by other threads of this CTA before the barrier; read them from the L2
        const unsigned long long e = GLOBAL ? __ldcg(buf + p) : buf[p];
        const int bk = bucket_of((unsigned)(e >> 32));
        const int s0 = start[bk], s1 = cur[bk];   // cur has advanced to the end of the bucket
        int rank = s0;
        for (int q = s0; q < s1; ++q) rank += (GLOBAL ? __ldcg(buf + q) : buf[q]) < e;
        out[rank] = (uint32_t)e;
    }
    __syncthreads();
    return true;
}

// =================================================================================================
// fused NMS kernel
// =================================================================================================
template <int K2_THREADS>
__global__ void __launch_bounds__(K2_THREADS, K2_THREADS == 512 ? NMS_MINB_512 : 1024 / K2_THREADS) nms_kernel(const __grid_constant__ K2Params P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int K = P.max_det;
    constexpr int WIN = K2_THREADS == 512 ? NMS_WIN_512 : K2_TAIL_WIN;
    // phase A: threads per candidate that share the walk over the cells under its box (the walks are chains of dependent
    // shared-memory loads: more, shorter chains as long as the CTA has the threads)
    constexpr int A_SUBS = K2_THREADS >= 512 ? A_SUBS_WIDE : 4;

    // ---- shared-memory carve-up (the sort's exchange buffer / sorted-index list overlays it)
    uint32_t *s_sidx = reinterpret_cast<uint32_t *>(smem_raw);
    float4 *s_sbox = reinterpret_cast<float4 *>(smem_raw + P.region0_bytes);                 // [WIN] window, NMS coordinates
    float4 *s_kbox = s_sbox + WIN;                                                           // [K] kept boxes
    // [K] (area bits, label, next kept box of the same cell, index into the filtered list): with the box, everything the
    // walk over a cell's list needs arrives in ONE round trip to shared memory (two 16-byte loads issued together)
    int4 *s_kmeta = reinterpret_cast<int4 *>(s_kbox + K);
    float2 *s_sctr = reinterpret_cast<float2 *>(s_kmeta + K);                                // [WIN] centres
    float *s_sarea = reinterpret_cast<float *>(s_sctr + WIN);                                // [WIN]
    float *s_sscore = s_sarea + WIN;                                                         // [WIN]
    int *s_slabel = reinterpret_cast<int *>(s_sscore + WIN);                                 // [WIN]
    int *s_sanchor = s_slabel + WIN;                                                         // [WIN]
    int *s_sorig = s_sanchor + WIN;                                                          // [WIN] index into the filtered list
    float *s_kscore = reinterpret_cast<float *>(s_sorig + WIN);                              // [K]
    int *s_kanchor = reinterpret_cast<int *>(s_kscore + K);                                  // [K]
    int *s_scell = s_kanchor + K;                                                            // [WIN] packed cell range under the box
    __shared__ unsigned int s_row32[NMS_CHUNK * 2];
    __shared__ int s_cellhead[MAX_CELLS], s_celltail[MAX_CELLS];
    __shared__ unsigned int s_supA[2];
    __shared__ unsigned char s_und[NMS_CHUNK];
    __shared__ int s_anyrow;
    __shared__ unsigned short s_pair[NMS_CHUNK * (NMS_CHUNK - 1) / 2];   // (i << 8) | j for every pair i < j of a chunk
    __shared__ unsigned long long s_keepm;

    BT_PHASE_INIT();
    // zero the per-image accumulators the mask kernel adds into
    if (tid < 8) P.acc[b * 8 + tid] = 0;
    if (tid == 10 && b == 0) *P.pool_used = 0ull;
    if (tid == 11 && b == 0) { P.n_items[0] = 0; P.n_items[1] = 0; }
    if (tid == 9 && P.seg_prob_sum) P.seg_prob_sum[b] = 0.0;
    if (tid == 12 && P.seg_soft2) { P.seg_soft2[2 * b] = 0; P.seg_soft2[2 * b + 1] = 0; }
    for (int i = tid; i < K; i += K2_THREADS) {
        if (P.inst_area) P.inst_area[(size_t)b * K + i] = 0;
        if (P.inst_inter) P.inst_inter[(size_t)b * K + i] = 0;
    }
    if (tid < MAX_CELLS) { s_cellhead[tid] = -1; s_celltail[tid] = -1; }
    if (tid >= 1 && tid < NMS_CHUNK)
        for (int i = 0; i < tid; ++i) s_pair[tid * (tid - 1) / 2 + i] = (unsigned short)((i << 8) | tid);
    const int M_all = P.n_cand[b];
    const float4 *cbox = P.cand_box + (size_t)b * P.cap;
    const float *cscore = P.cand_score + (size_t)b * P.cap;
    const int32_t *clabel = P.cand_label + (size_t)b * P.cap;
    const int32_t *canchor = P.cand_anchor + (size_t)b * P.cap;

    // ---- 1. stable descending sort: key = (descending score key << 32) | candidate index
    const unsigned long long *gkeys = nullptr;
    const uint32_t *gidx = nullptr;   // long lists sorted by the bucket sort: index list in the workspace
    bool sorted = false;
    {
        unsigned long long *s_x = reinterpret_cast<unsigned long long *>(smem_raw);
        const int Mp_all = (M_all + 31) & ~31;
        unsigned long long *gslice = P.sort_keys + (size_t)b * P.sort_stride;
        unsigned long long *sbuf = reinterpret_cast<unsigned long long *>(smem_raw + P.region0_bytes);
        if (M_all <= P.bucket_max) sorted = bucket_sort<K2_THREADS, false>(cscore, M_all, sbuf, reinterpret_cast<int *>(sbuf + Mp_all), s_sidx);
        else {
            sorted = bucket_sort<K2_THREADS, true>(cscore, M_all, gslice, reinterpret_cast<int *>(sbuf), reinterpret_cast<uint32_t *>(gslice + Mp_all));
            if (sorted) gidx = reinterpret_cast<const uint32_t *>(gslice + Mp_all);
        }
        if (sorted) {
        } else if (M_all <= RADIX_MAX) radix_sort_to_smem<K2_THREADS>(cscore, M_all, smem_raw, s_sidx);
        else if (K2_THREADS == 256 && M_all <= 256) sort_to_smem<1>(cscore, M_all, 256, s_x, s_sidx);
        else if (K2_THREADS == 256 && M_all <= 512) sort_to_smem<2>(cscore, M_all, 256, s_x, s_sidx);
        else if (K2_THREADS == 256 && M_all <= 1024) sort_to_smem<4>(cscore, M_all, 256, s_x, s_sidx);
        else if (K2_THREADS == 256 && M_all <= 2048) sort_to_smem<8>(cscore, M_all, 256, s_x, s_sidx);
        else if (K2_THREADS == 256 && M_all <= SORT_SMALL_MAX) sort_to_smem<16>(cscore, M_all, 256, s_x, s_sidx);
        else if (K2_THREADS == 512 && M_all <= 512) sort_to_smem<1>(cscore, M_all, 512, s_x, s_sidx);
        else if (K2_THREADS == 512 && M_all <= 1024) sort_to_smem<2>(cscore, M_all, 512, s_x, s_sidx);
        else if (K2_THREADS == 512 && M_all <= 2048) sort_to_smem<4>(cscore, M_all, 512, s_x, s_sidx);
        else if (K2_THREADS == 512 && M_all <= SORT_SMALL_MAX) sort_to_smem<8>(cscore, M_all, 512, s_x, s_sidx);
        else if (K2_THREADS == 1024 && M_all <= 1024) sort_to_smem<1>(cscore, M_all, 1024, s_x, s_sidx);
        else if (K2_THREADS == 1024 && M_all <= 2048) sort_to_smem<2>(cscore, M_all, 1024, s_x, s_sidx);
        else if (K2_THREADS == 1024 && M_all <= 4096) sort_to_smem<4>(cscore, M_all, 1024, s_x, s_sidx);
        else if (K2_THREADS == 1024 && M_all <= 8192) sort_to_smem<16>(cscore, M_all, 512, s_x, s_sidx);
        else if (K2_THREADS == 1024 && M_all <= SORT_REG_MAX) sort_to_smem<16>(cscore, M_all, 1024, s_x, s_sidx);
        else {
            // very long lists (30k-candidate stress case): bitonic network in global memory
            int P2 = 1;
            while (P2 < M_all) P2 <<= 1;
            unsigned long long *keys = gslice;
            for (int i = tid; i < P2; i += K2_THREADS)
                keys[i] = (i < M_all) ? (((unsigned long long)desc_key(cscore[i]) << 32) | (unsigned)i) : ~0ull;
            __syncthreads();
            for (int k = 2; k <= P2; k <<= 1)
                for (int j = k >> 1; j > 0; j >>= 1) {
                    for (int t = tid; t < (P2 >> 1); t += K2_THREADS) {
                        int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                        int l = i | j;
                        unsigned long long a = keys[i], c = keys[l];
                        bool asc = (i & k) == 0;
                        if ((a > c) == asc) { keys[i] = c; keys[l] = a; }
                    }
                    __syncthreads();
                }
            gkeys = keys;
        }
    }
    BT_PHASE_MARK(1, 0);   // sort
    const int M = min(M_all, P.limit);   // Ultralytics max_nms: only the best `limit` candidates enter the sweep

    auto cell_x = [&](float x) { return min(max(__float2int_rd(__fmul_rn(x, P.inv_cw)), 0), P.gx - 1); };
    auto cell_y = [&](float y) { return min(max(__float2int_rd(__fmul_rn(y, P.inv_ch)), 0), P.gy - 1); };

    // ---- 2. greedy sweep over windows of 1024 sorted candidates, 64 at a time
    int nkept = 0;
    for (int w0 = 0; w0 < M && nkept < K; w0 += WIN) {
        const int wn = min(WIN, M - w0);
        // (a) stage the window in NMS order; bucket its candidates by the cell of their centre
        for (int t = tid; t < wn; t += K2_THREADS) {
            const int idx = gidx ? (int)__ldcg(gidx + w0 + t) : gkeys ? (int)(unsigned)gkeys[w0 + t] : (int)s_sidx[w0 + t];
            float4 bx = __ldg(cbox + idx);
            const int lb = __ldg(clabel + idx);
            s_sscore[t] = __ldg(cscore + idx);
            s_sanchor[t] = __ldg(canchor + idx);
            s_sorig[t] = idx;
            if (P.class_mode == BT_CLASS_OFFSET) {
                const float off = __fmul_rn((float)lb, P.max_wh);
                bx.x = __fadd_rn(bx.x, off); bx.y = __fadd_rn(bx.y, off);
                bx.z = __fadd_rn(bx.z, off); bx.w = __fadd_rn(bx.w, off);
            }
            s_sbox[t] = bx;
            s_sctr[t] = make_float2(__fmul_rn(__fadd_rn(bx.x, bx.z), 0.5f), __fmul_rn(__fadd_rn(bx.y, bx.w), 0.5f));
            {   // cells under the box: x0 | y0 << 4 | nx << 8 | ny << 13 (nx = 1, ny = 0 for an inverted box)
                const int gx0 = cell_x(bx.x), gy0 = cell_y(bx.y);
                const int ncx = max(cell_x(bx.z) - gx0 + 1, 1), ncy = max(cell_y(bx.w) - gy0 + 1, 0);
                s_scell[t] = gx0 | (gy0 << 4) | (ncx << 8) | (ncy << 13);
            }
            s_sarea[t] = box_area(bx);
            s_slabel[t] = lb;
        }
        __syncthreads();
        BT_PHASE_MARK(1, 1);   // stage window
        // (c) the chunks, in order
        for (int c0 = 0; c0 < wn && nkept < K; c0 += NMS_CHUNK) {
            const int n_in = min(NMS_CHUNK, wn - c0);
            if (tid < 2 * NMS_CHUNK) s_row32[tid] = 0;
            if (tid < 2) s_supA[tid] = 0;
            if (tid == 2) s_anyrow = 0;
            __syncthreads();
            // (A) chunk vs kept boxes.  Centre-cull mode: only kept boxes whose centre lies in a cell under
            // the candidate's box can suppress it; 4 threads per candidate walk those cells (8 warps: the
            // phase is issue-bound, r01k).  Otherwise 16 threads per candidate stride over all kept boxes.
            if (P.centre_cull) {
                if (tid < A_SUBS * NMS_CHUNK) {
                    const int ci = tid / A_SUBS, sub = tid % A_SUBS;
                    bool f = false;
                    if (ci < n_in) {
                        const float4 bj = s_sbox[c0 + ci];
                        const float2 cj = s_sctr[c0 + ci];
                        const float aj = s_sarea[c0 + ci];
                        const int lj = s_slabel[c0 + ci];
                        const int pc = s_scell[c0 + ci];
                        const int gx0 = pc & 15, gy0 = (pc >> 4) & 15, ncx = (pc >> 8) & 31, ncy = (pc >> 13) & 31;
                        // cells sub, sub + A_SUBS, ... in row-major order (1 <= ncx <= 16): row = floor(cell / ncx) from a float
                        // product ((cell + 0.5) / ncx is at least 1/32 away from an integer; stepping qx down by ncx cost 11 %
                        // of the kernel's instructions, r02c)
                        const float inv_ncx = __frcp_rn((float)ncx);
                        int cell = sub;
                        int qy = __float2int_rz(__fmul_rn((float)cell + 0.5f, inv_ncx)), qx = cell - qy * ncx;
                        while (qy < ncy && !f) {
                            // lists are in keep order: the strongest box of a cluster comes first and usually settles it
                            for (int k = s_cellhead[(gy0 + qy) * P.gx + gx0 + qx]; k >= 0 && !f;) {
                                const float4 kb = s_kbox[k];
                                const int4 km = s_kmeta[k];
                                k = km.z;
                                // the kept box's centre, the expression its cell was chosen by
                                const float ckx = __fmul_rn(__fadd_rn(kb.x, kb.z), 0.5f), cky = __fmul_rn(__fadd_rn(kb.y, kb.w), 0.5f);
                                if (!(ckx >= bj.x && ckx <= bj.z && cky >= bj.y && cky <= bj.w)) continue;
                                f = suppresses(kb, __int_as_float(km.x), km.y, bj, aj, lj, P.thr_up, P.early_out, P.class_mode, 1,
                                               cj.x, cj.y, P.fast);
                            }
                            cell += A_SUBS;
                            qy = __float2int_rz(__fmul_rn((float)cell + 0.5f, inv_ncx));
                            qx = cell - qy * ncx;
                        }
                    }
                    const unsigned m = __ballot_sync(0xffffffffu, f);
                    if ((lane & (A_SUBS - 1)) == 0 && ((m >> lane) & ((1u << A_SUBS) - 1u))) atomicOr(&s_supA[ci >> 5], 1u << (ci & 31));
                }
            } else {
                for (int ci = tid >> 4; ci < NMS_CHUNK; ci += K2_THREADS >> 4) {   // warp-uniform trip count
                    const int sub = tid & 15;
                    bool f = false;
                    if (ci < n_in) {
                        const float4 bj = s_sbox[c0 + ci];
                        const float aj = s_sarea[c0 + ci];
                        const int lj = s_slabel[c0 + ci];
                        for (int k = sub; k < nkept && !f; k += 16) {
                            const int4 km = s_kmeta[k];
                            f = suppresses(s_kbox[k], __int_as_float(km.x), km.y, bj, aj, lj, P.thr_up, P.early_out, P.class_mode, 0,
                                           0.0f, 0.0f, P.fast);
                        }
                    }
                    const unsigned m = __ballot_sync(0xffffffffu, f);
                    if ((lane & 15) == 0 && ((m >> lane) & 0xffffu)) atomicOr(&s_supA[ci >> 5], 1u << (ci & 31));
                }
            }
            __syncthreads();
            BT_PHASE_MARK(1, 8);   // chunk: A
            // (B) "who suppresses me" rows of the candidates A left undecided, against the undecided
            // earlier candidates of the chunk only (a cluster of hundreds of candidates on one object is
            // settled by A as soon as its leader is kept).  One thread per pair (i < j) of the chunk, from a
            // table of the 2016 pairs; the exact IoU runs only for pairs that pass the cheap necessary test.
            const unsigned long long valid = (n_in == 64) ? ~0ull : ((1ull << n_in) - 1ull);
            const unsigned long long und0 = valid & ~(((unsigned long long)s_supA[1] << 32) | s_supA[0]);
            // Only the pairs of UNDECIDED candidates are enumerated: every warp compacts the undecided set into the same
            // 64-byte table (identical values from every warp: no block barrier), pair number pq of the triangular table
            // then names two table positions.  Usually one trip per thread instead of 2016 / threads.
            const int n_und = __popcll(und0);
            {
                const unsigned ulo = (unsigned)und0, uhi = (unsigned)(und0 >> 32), ltm = (1u << lane) - 1u;
                if ((ulo >> lane) & 1u) s_und[__popc(ulo & ltm)] = (unsigned char)lane;
                if ((uhi >> lane) & 1u) s_und[__popc(ulo) + __popc(uhi & ltm)] = (unsigned char)(lane + 32);
                __syncwarp();
            }
            for (int pq = tid; pq < n_und * (n_und - 1) / 2; pq += K2_THREADS) {
                const int pr = s_pair[pq], io = s_und[pr >> 8], jo = s_und[pr & 255];
                const int i = c0 + io, j = c0 + jo;
                const float4 bi = s_sbox[i], bj = s_sbox[j];
                const float2 cj = s_sctr[j];
                if (P.centre_cull) {
                    const float2 ci = s_sctr[i];
                    if (!(ci.x >= bj.x && ci.x <= bj.z && ci.y >= bj.y && ci.y <= bj.w && cj.x >= bi.x && cj.x <= bi.z &&
                          cj.y >= bi.y && cj.y <= bi.w))
                        continue;
                } else if (P.early_out) {
                    if (!(fminf(bi.z, bj.z) > fmaxf(bi.x, bj.x) && fminf(bi.w, bj.w) > fmaxf(bi.y, bj.y))) continue;
                }
                if (suppresses(bi, s_sarea[i], s_slabel[i], bj, s_sarea[j], s_slabel[j], P.thr_up, P.early_out, P.class_mode,
                               P.centre_cull, cj.x, cj.y, P.fast)) {
                    atomicOr(&s_row32[jo * 2 + (io >> 5)], 1u << (io & 31));
                    s_anyrow = 1;
                }
            }
            __syncthreads();
            BT_PHASE_MARK(1, 11);  // chunk: B
            unsigned long long keepm;
            if (s_anyrow) {
                // (C) one warp resolves the chunk as a fixpoint over the rows (lane: rows lane, lane + 32)
                if (wid == 0) {
                    const unsigned long long row_a = ((unsigned long long)s_row32[lane * 2 + 1] << 32) | s_row32[lane * 2];
                    const unsigned long long row_b = ((unsigned long long)s_row32[(lane + 32) * 2 + 1] << 32) | s_row32[(lane + 32) * 2];
                    unsigned long long und = und0, km = 0ull;
                    while (und) {
                        // kept: no undecided and no kept suppressor left; removed: a kept suppressor exists
                        const bool ua = (und >> lane) & 1ull, ub = (und >> (lane + 32)) & 1ull;
                        const unsigned long long live = und | km;
                        const unsigned long long newk =
                            ((unsigned long long)__ballot_sync(0xffffffffu, ub && (row_b & live) == 0ull) << 32) |
                            __ballot_sync(0xffffffffu, ua && (row_a & live) == 0ull);
                        km |= newk;
                        und &= ~newk;
                        const unsigned long long rem =
                            ((unsigned long long)__ballot_sync(0xffffffffu, ub && (row_b & km) != 0ull) << 32) |
                            __ballot_sync(0xffffffffu, ua && (row_a & km) != 0ull);
                        und &= ~rem;
                    }
                    if (lane == 0) s_keepm = km;
                }
                __syncthreads();
                keepm = s_keepm;
            } else {
                keepm = und0;   // nobody in the chunk suppresses anybody: every undecided candidate is kept
            }
            {
                // [:TOP_K]: only the first `room` keeps survive (later ones cannot affect earlier ones)
                const int room = K - nkept;
                if (__popcll(keepm) > room) {   // room < 64 here: cut after the room-th set bit
                    const unsigned lo = (unsigned)keepm, hi = (unsigned)(keepm >> 32);
                    const int nlo = __popc(lo);
                    if (room == 0) keepm = 0ull;
                    else if (room <= nlo) keepm &= (2ull << __fns(lo, 0, room)) - 1ull;
                    else keepm &= (2ull << (32 + __fns(hi, 0, room - nlo))) - 1ull;
                }
            }
            BT_PHASE_MARK(1, 9);   // chunk: C
            if (tid < NMS_CHUNK && ((keepm >> tid) & 1ull)) {
                const int slot = nkept + __popcll(keepm & ((1ull << tid) - 1ull));
                const float2 ctr = s_sctr[c0 + tid];
                s_kbox[slot] = s_sbox[c0 + tid];
                s_kmeta[slot] = make_int4(__float_as_int(s_sarea[c0 + tid]), s_slabel[c0 + tid], -1, s_sorig[c0 + tid]);
                s_kscore[slot] = s_sscore[c0 + tid];
                s_kanchor[slot] = s_sanchor[c0 + tid];
                if (P.centre_cull) {
                    // append to the cell's list (keep order: earlier, stronger boxes first)
                    const int cell = cell_y(ctr.y) * P.gx + cell_x(ctr.x);
                    const int prev = atomicExch(&s_celltail[cell], slot);
                    if (prev < 0) s_cellhead[cell] = slot; else s_kmeta[prev].z = slot;
                }
            }
            nkept += __popcll(keepm);
            BT_PHASE_MARK(1, 10);  // chunk: insert
        }
        __syncthreads();   // the window is re-staged next
        BT_PHASE_MARK(1, 3);   // chunks
    }

    // ---- 3. package kept detections (running_main_v2.py:818-839); zero-fill the padding
    if (tid == 0) P.det_count[b] = nkept;
    for (int k = tid; k < K; k += K2_THREADS) {
        float *o = P.dets + ((size_t)b * K + k) * 6;
        if (k < nkept) {
            const int4 km = s_kmeta[k];
            const int idx = km.w;
            float4 bx = s_kbox[k];
            if (P.class_mode == BT_CLASS_OFFSET) bx = __ldg(cbox + idx);   // un-offset coordinates
            o[0] = bx.x; o[1] = bx.y; o[2] = bx.z; o[3] = bx.w;
            o[4] = s_kscore[k];
            o[5] = (float)km.y;
            P.det_keep[(size_t)b * K + k] = idx;
            P.det_anchor[(size_t)b * K + k] = s_kanchor[k];
            int r_lo, r_hi, c_lo, c_hi;
            const float bb[4] = {bx.x, bx.y, bx.z, bx.w};
            const bool ok = crop_region(bb, P.crop, P.rx, P.ry, P.PW, P.PH, r_lo, r_hi, c_lo, c_hi);
            P.det_region[(size_t)b * K + k] = ok ? make_short4((short)r_lo, (short)r_hi, (short)c_lo, (short)c_hi)
                                                 : make_short4(1, 0, 1, 0);
        } else {
            P.det_region[(size_t)b * K + k] = make_short4(1, 0, 1, 0);
            o[0] = o[1] = o[2] = o[3] = o[4] = o[5] = 0.0f;
            P.det_keep[(size_t)b * K + k] = -1;
            P.det_anchor[(size_t)b * K + k] = -1;
        }
    }
    // clear the matching table (filled by match_kernel)
    if (P.dt_match) {
        const size_t per_img = (size_t)BT_NUM_AREA * P.T * K;
        int32_t *dm = P.dt_match + (size_t)b * per_img;
        if ((per_img & 3) == 0) {
            int4 *d4 = reinterpret_cast<int4 *>(dm);   // per-image base is 16-byte aligned when per_img % 4 == 0
            for (int q = tid; q < (int)(per_img >> 2); q += K2_THREADS) d4[q] = make_int4(0, 0, 0, 0);
        } else {
            for (int q = tid; q < (int)per_img; q += K2_THREADS) dm[q] = 0;
        }
    }
    BT_PHASE_MARK(1, 6);   // package
}

// =================================================================================================
// mask-coefficient gather, spread over the whole GPU: 8 detections x 32 coefficients per CTA
// =================================================================================================
__global__ void __launch_bounds__(GM_THREADS) coeff_gather_kernel(const __grid_constant__ K2Params P) {
    const int b = blockIdx.y, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int K = P.max_det;
    const int k = blockIdx.x * 8 + wid, m = lane;
    if (k < K) {
        const int a = P.det_anchor[(size_t)b * K + k];
        float v = 0.0f;
        if (a >= 0) {
            if (P.head_bf16) {
                const unsigned short *src = (P.layout == BT_LAYOUT_L2)
                                                ? static_cast<const unsigned short *>(P.head) + ((size_t)b * P.C + 4 + P.nc) * P.N
                                                : static_cast<const unsigned short *>(P.coeffs) + (size_t)b * P.nm * P.N;
                v = __uint_as_float((unsigned)__ldg(src + (size_t)m * P.N + a) << 16);
            } else {
                const float *src = (P.layout == BT_LAYOUT_L2) ? static_cast<const float *>(P.head) + ((size_t)b * P.C + 4 + P.nc) * P.N
                                                              : static_cast<const float *>(P.coeffs) + (size_t)b * P.nm * P.N;
                v = __ldg(src + (size_t)m * P.N + a);   // nm == 32 (validated by check_params)
            }
        }
        P.det_coeff[((size_t)b * K + k) * 32 + m] = v;
    }
}

// =================================================================================================
// plan of the mask stage, one CTA per image: where each detection's crop-box logits live in the pool (exclusive
// prefix sum of the box areas; the image's base comes from one bump of the pool counter), which contract_kernel
// tiles each detection touches, and the work items of cells_kernel.  Independent of the coefficient gather.
// =================================================================================================
__global__ void __launch_bounds__(GM_THREADS) plan_kernel(const __grid_constant__ K2Params P) {
    const int b = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int K = P.max_det;
    __shared__ long long s_base;
    const int tid = threadIdx.x;
    const int per = (K + GM_THREADS - 1) / GM_THREADS;
    const short4 *reg = P.det_region + (size_t)b * K;
    auto chunks_of = [](const short4 &rg) {   // 2x2 cell blocks under the crop box, in chunks of C_CHUNK
        const int nb = (((rg.w + 1) >> 1) - (rg.z >> 1) + 1) * (((rg.y + 1) >> 1) - (rg.x >> 1) + 1);
        return (nb + C_CHUNK - 1) / C_CHUNK;
    };
    int mine = 0, mych = 0;
    for (int i = 0; i < per; ++i) {
        const int kk = tid * per + i;
        if (kk < K) {
            const short4 rg = reg[kk];
            if (rg.x <= rg.y && rg.z <= rg.w) { mine += (rg.y - rg.x + 1) * (rg.w - rg.z + 1); mych += chunks_of(rg); }
        }
    }
    // a full-image box is < 2^16 * 2^16; the running sum is kept in 64 bits only across warps
    long long incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long u = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += u;
    }
    int cincl = mych;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, cincl, d);
        if (lane >= d) cincl += u;
    }
    __shared__ long long s_wtot[GM_THREADS / 32];
    __shared__ int s_ctot[GM_THREADS / 32], s_ibase;
    if (lane == 31) { s_wtot[wid] = incl; s_ctot[wid] = cincl; }
    __syncthreads();
    long long before = 0, total = 0;
    int cbefore = 0, ctotal = 0;
    for (int w = 0; w < GM_THREADS / 32; ++w) {
        const long long v = s_wtot[w]; if (w < wid) before += v; total += v;
        const int c = s_ctot[w]; if (w < wid) cbefore += c; ctotal += c;
    }
    if (tid == 0) {
        // the counter saturates instead of wrapping: images that find the pool full use no pool at all
        const long long want = total > P.pool_cap ? P.pool_cap : total;
        s_base = (long long)atomicAdd(reinterpret_cast<unsigned long long *>(P.pool_used), (unsigned long long)want);
        s_ibase = atomicAdd(P.n_items, ctotal);
    }
    __syncthreads();
    long long off = s_base + before + incl - mine;
    for (int i = 0; i < per; ++i) {
        const int kk = tid * per + i;
        if (kk < K) {
            const short4 rg = reg[kk];
            int o = -1;
            if (rg.x <= rg.y && rg.z <= rg.w) {
                const long long area = (long long)(rg.y - rg.x + 1) * (rg.w - rg.z + 1);
                if (off + area <= P.pool_cap) o = (int)off;
                else P.n_items[1] = 1;   // cells_kernel will read prototypes itself: contract_kernel keeps them in the L2
                off += area;
            }
            P.scr_off[(size_t)b * K + kk] = o;
        }
    }
    // tile lists of contract_kernel: every detection with pool room goes into the tiles its crop box touches
    __shared__ int s_tcnt[PLAN_MAX_TILES];
    for (int t = tid; t < P.ntiles; t += GM_THREADS) s_tcnt[t] = 0;
    __syncthreads();
    {
        long long off2 = s_base + before + incl - mine;
        for (int i = 0; i < per; ++i) {
            const int kk = tid * per + i;
            if (kk < K) {
                const short4 rg = reg[kk];
                if (rg.x <= rg.y && rg.z <= rg.w) {
                    const long long area = (long long)(rg.y - rg.x + 1) * (rg.w - rg.z + 1);
                    if (off2 + area <= P.pool_cap) {
                        for (int ty = rg.x / TA_H; ty <= rg.y / TA_H; ++ty)
                            for (int tx = rg.z / TA_W; tx <= rg.w / TA_W; ++tx) {
                                const int t = ty * P.ntx + tx;
                                P.tile_list[((size_t)b * P.ntiles + t) * K + atomicAdd(&s_tcnt[t], 1)] = (unsigned short)kk;
                            }
                    }
                    off2 += area;
                }
            }
        }
    }
    __syncthreads();
    for (int t = tid; t < P.ntiles; t += GM_THREADS) P.tile_cnt[(size_t)b * P.ntiles + t] = s_tcnt[t];
    // work items of cells_kernel (any order; the capacity covers every detection at full-image size)
    int ci = s_ibase + cbefore + cincl - mych;
    for (int i = 0; i < per; ++i) {
        const int kk = tid * per + i;
        if (kk < K) {
            const short4 rg = reg[kk];
            if (rg.x <= rg.y && rg.z <= rg.w) {
                const int nc = chunks_of(rg);
                for (int c = 0; c < nc; ++c, ++ci)
                    if (ci < P.item_cap) P.items[ci] = make_int2(b * K + kk, c);
            }
        }
    }
}

// =================================================================================================
// COCOeval.evaluateImg (one CTA per image)
// =================================================================================================
__global__ void __launch_bounds__(GM_THREADS) match_kernel(const __grid_constant__ K2Params P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int K = P.max_det;
    if (P.dt_match == nullptr) return;
    BT_PHASE_INIT();
    // ---- COCOeval.evaluateImg for every (class, area range, IoU threshold)
    const int G = P.gt_count[b];
    const int D = P.det_count[b];
    const int T = P.T;
    double *s_db = reinterpret_cast<double *>(smem_raw);   // [K][4] x, y, w, h
    double *s_gb = s_db + (size_t)K * 4;                   // [max_gt][4]
    double *s_iou = s_gb + (size_t)P.max_gt * 4;           // [D][G] if it fits
    const int iou_room = P.coco_smem_doubles - K * 4 - P.max_gt * 4;
    const bool iou_in_smem = (D * G) <= iou_room;
    int *s_dl = reinterpret_cast<int *>(s_db + P.coco_smem_doubles);   // [K] det labels
    int *s_can = s_dl + K;                                              // [K] 1 if the det can match at the loosest threshold
    int *s_list = s_can + K;                                            // [K] compacted list of those dets
    // [K] match bits per detection (bit a * T + t) and "matched to an ignored GT" bits, for the sweep records
    unsigned long long *s_mbits = reinterpret_cast<unsigned long long *>(s_list + K + (K & 1));
    unsigned long long *s_gibits = s_mbits + K;
    __shared__ int s_gl[32];
    __shared__ unsigned s_gign[BT_NUM_AREA];
    __shared__ int s_warpcnt[GM_THREADS / 32];
    __shared__ int s_nlist;

    for (int k = tid; k < D; k += GM_THREADS) {
        s_mbits[k] = 0ull; s_gibits[k] = 0ull;
        const float *o = P.dets + ((size_t)b * K + k) * 6;
        s_db[k * 4 + 0] = (double)o[0];
        s_db[k * 4 + 1] = (double)o[1];
        s_db[k * 4 + 2] = (double)__fsub_rn(o[2], o[0]);
        s_db[k * 4 + 3] = (double)__fsub_rn(o[3], o[1]);
        s_dl[k] = (int)o[5];
    }
    if (tid < G) {
        const float *g = P.gt_boxes + ((size_t)b * P.max_gt + tid) * 4;
        s_gb[tid * 4 + 0] = (double)g[0];
        s_gb[tid * 4 + 1] = (double)g[1];
        s_gb[tid * 4 + 2] = (double)__fsub_rn(g[2], g[0]);
        s_gb[tid * 4 + 3] = (double)__fsub_rn(g[3], g[1]);
        s_gl[tid] = P.gt_labels[(size_t)b * P.max_gt + tid];
    }
    __syncthreads();
    const double area_lo[BT_NUM_AREA] = COCO_AREA_LO;
    const double area_hi[BT_NUM_AREA] = COCO_AREA_HI;
    if (tid < BT_NUM_AREA) {
        unsigned m = 0;
        for (int g = 0; g < G; ++g) {
            double ar = s_gb[g * 4 + 2] * s_gb[g * 4 + 3];
            bool in_cls = s_gl[g] >= 0 && s_gl[g] < P.nc;
            bool ig = in_cls && (ar < area_lo[tid] || ar > area_hi[tid]);
            if (ig) m |= 1u << g;
            if (P.gt_ignore) P.gt_ignore[((size_t)b * BT_NUM_AREA + tid) * P.max_gt + g] = ig ? 1 : 0;
        }
        for (int g = G; g < P.max_gt; ++g)
            if (P.gt_ignore) P.gt_ignore[((size_t)b * BT_NUM_AREA + tid) * P.max_gt + g] = 0;
        s_gign[tid] = m;
    }
    // IoU table + per-detection best IoU over same-class GT
    double thr_min = 1.0;
    for (int t = 0; t < T; ++t) thr_min = fmin(thr_min, fmin(P.thrs[t], 1 - 1e-10));
    for (int k = tid; k < D; k += GM_THREADS) {
        double best = -1.0;
        for (int g = 0; g < G; ++g) {
            double v = bb_iou(s_db + k * 4, s_gb + g * 4);
            if (iou_in_smem) s_iou[k * G + g] = v;
            if (s_gl[g] == s_dl[k] && v > best) best = v;
        }
        s_can[k] = (best >= thr_min) ? 1 : 0;
    }
    // default (unmatched) ignore flags for every (a, t, d), zero padding beyond D
    if (P.dt_ignore) {
        const size_t per_img = (size_t)BT_NUM_AREA * T * K;
        uint8_t *di = P.dt_ignore + (size_t)b * per_img;
        for (int d = tid; d < K; d += GM_THREADS) {
            unsigned igm = 0;
            if (d < D) {
                const double ar = s_db[d * 4 + 2] * s_db[d * 4 + 3];
#pragma unroll
                for (int a = 0; a < BT_NUM_AREA; ++a) igm |= ((ar < area_lo[a] || ar > area_hi[a]) ? 1u : 0u) << a;
            }
            for (int a = 0; a < BT_NUM_AREA; ++a)
                for (int t = 0; t < T; ++t) di[((size_t)a * T + t) * K + d] = (igm >> a) & 1u;
        }
    }
    __syncthreads();
    // ordered compaction of the detections that can match at the loosest threshold
    {
        int base = 0;
        for (int k0 = 0; k0 < D; k0 += GM_THREADS) {
            int k = k0 + tid;
            bool f = (k < D) && s_can[k] != 0;
            unsigned m = __ballot_sync(0xffffffffu, f);
            if (lane == 0) s_warpcnt[wid] = __popc(m);
            __syncthreads();
            int off = base, tot = 0;
            for (int w = 0; w < GM_THREADS / 32; ++w) { int v = s_warpcnt[w]; if (w < wid) off += v; tot += v; }
            __syncthreads();
            if (f) s_list[off + __popc(m & ((1u << lane) - 1u))] = k;
            base += tot;
        }
        if (tid == 0) s_nlist = base;
        __syncthreads();
    }
    // greedy matching, one thread per (area range, threshold), over the compacted list only
    if (tid < BT_NUM_AREA * T) {
        const int a = tid / T, t = tid - a * T;
        const unsigned gign = s_gign[a];
        unsigned gm = 0;
        const double thr = fmin(P.thrs[t], 1 - 1e-10);
        const int nl = s_nlist;
        for (int li = 0; li < nl; ++li) {
            const int d = s_list[li];
            const int dl = s_dl[d];
            double best = thr;
            int m = -1;
            for (int pass = 0; pass < 2; ++pass) {
                if (pass == 1 && m >= 0) break;          // matched a regular GT: stop at the first ignored one
                for (int g = 0; g < G; ++g) {
                    if ((((gign >> g) & 1u) != 0) != (pass == 1)) continue;
                    if ((gm >> g) & 1u) continue;
                    if (s_gl[g] != dl) continue;
                    double v = iou_in_smem ? s_iou[d * G + g] : bb_iou(s_db + d * 4, s_gb + g * 4);
                    if (v < best) continue;
                    best = v;
                    m = g;
                }
            }
            if (m >= 0) {
                gm |= 1u << m;
                size_t o = (((size_t)b * BT_NUM_AREA + a) * T + t) * K + d;
                P.dt_match[o] = m + 1;
                if (P.dt_ignore) P.dt_ignore[o] = (gign >> m) & 1u;
                if (P.sweep) {
                    atomicOr(&s_mbits[d], 1ull << tid);
                    if ((gign >> m) & 1u) atomicOr(&s_gibits[d], 1ull << tid);
                }
            }
        }
    }
    BT_PHASE_MARK(1, 7);   // COCO matching
    // ---- sweep records (a9): what torchmetrics keeps per image for COCOeval.accumulate, appended on the device
    if (P.sweep) {
        __syncthreads();
        long long *hdr = P.sweep;
        BtSweepRecord *ring = reinterpret_cast<BtSweepRecord *>(hdr + BT_SWEEP_HEADER_I64);
        __shared__ long long s_rbase, s_rcap;
        if (tid == 0) {
            atomicAdd(reinterpret_cast<unsigned long long *>(hdr + BT_SWEEP_N_IMAGES), 1ull);
            s_rbase = D ? (long long)atomicAdd(reinterpret_cast<unsigned long long *>(hdr + BT_SWEEP_N_RECORDS), (unsigned long long)D) : 0;
            s_rcap = hdr[BT_SWEEP_CAPACITY];
        }
        // non-ignored GT per (area range, class); v2 drops the target of an image without candidates (running_main_v2.py:797-814)
        if (!(P.drop_gt_no_cand && P.n_cand[b] == 0)) {
            for (int q = tid; q < BT_NUM_AREA * P.nc; q += GM_THREADS) {
                const int a = q / P.nc, c = q - a * P.nc;
                int cnt = 0;
                for (int g = 0; g < G; ++g) cnt += (s_gl[g] == c && !((s_gign[a] >> g) & 1u)) ? 1 : 0;
                if (cnt) atomicAdd(reinterpret_cast<unsigned long long *>(hdr + BT_SWEEP_NPIG + a * BT_MAX_CLASSES + c), (unsigned long long)cnt);
            }
        }
        __syncthreads();
        const unsigned long long tmask = (T >= 16) ? 0xffffull : ((1ull << T) - 1ull);
        for (int d = tid; d < D; d += GM_THREADS) {
            const long long pos = s_rbase + d;
            if (pos >= s_rcap) continue;   // ring full: reported through the header (N_RECORDS > CAPACITY)
            const int lab = s_dl[d];
            int cr = 0;
            for (int j = 0; j < d; ++j) cr += (s_dl[j] == lab) ? 1 : 0;
            const double ar = s_db[d * 4 + 2] * s_db[d * 4 + 3];
            unsigned long long amask = 0ull;   // unmatched detections outside the area range are ignored
#pragma unroll
            for (int a = 0; a < BT_NUM_AREA; ++a)
                if (ar < area_lo[a] || ar > area_hi[a]) amask |= tmask << (a * T);
            const unsigned long long mb = s_mbits[d];
            BtSweepRecord r;
            r.matched = mb;
            r.ignored = s_gibits[d] | (~mb & amask);
            r.score_key = desc_key(P.dets[((size_t)b * K + d) * 6 + 4]);
            r.image = (uint32_t)(P.image_offset + (P.image_base ? __ldg(P.image_base) : 0) + b);
            r.rank = (uint16_t)d;
            r.class_rank = (uint16_t)cr;
            r.label = (uint8_t)lab;
            r.pad[0] = r.pad[1] = r.pad[2] = 0;
            uint4 *dst = reinterpret_cast<uint4 *>(ring + pos);
            const uint4 *src = reinterpret_cast<const uint4 *>(&r);
            dst[0] = src[0];
            dst[1] = src[1];
        }
    }
}

int launch_nms_match(const BtParams &p, const BtIO &io, const Workspace &w, cudaStream_t s, int parts) {
    K2Params P{};
    P.N = p.num_anchors; P.nc = p.nc; P.nm = p.nm; P.C = 4 + p.nc + p.nm;
    P.cap = cand_capacity(&p); P.cap_pow2 = next_pow2(P.cap); P.limit = cand_limit(&p);
    P.max_det = p.max_det; P.max_gt = p.max_gt; P.class_mode = p.class_mode; P.layout = p.layout;
    float t = (float)p.iou_thres;
    if (!((double)t > p.iou_thres)) t = nextafterf(t, INFINITY);
    P.thr_up = t;
    P.fast.on = t >= 1e-3f ? 1 : 0;
    P.fast.lo = (float)((double)t * (1.0 - 1e-6));
    P.fast.hi = (float)((double)t * (1.0 + 1e-6));
    P.early_out = p.iou_thres >= 0.0 ? 1 : 0;
    P.max_wh = p.max_wh;
    P.head = io.head; P.head_bf16 = p.head_dtype == BT_HEAD_BF16; P.coeffs = io.coeffs;
    P.cand_box = w.cand_box; P.cand_score = w.cand_score; P.cand_label = w.cand_label;
    P.cand_anchor = w.cand_anchor; P.n_cand = io.n_cand; P.sort_keys = w.sort_keys;
    P.det_count = io.det_count; P.dets = io.dets; P.det_keep = io.det_keep;
    P.det_anchor = io.det_anchor; P.det_coeff = io.det_coeff;
    P.gt_count = io.gt_count; P.gt_boxes = io.gt_boxes; P.gt_labels = io.gt_labels;
    P.T = p.num_iou_thrs;
    for (int i = 0; i < p.num_iou_thrs; ++i) P.thrs[i] = p.iou_thrs[i];
    P.dt_match = io.dt_match; P.dt_ignore = io.dt_ignore; P.gt_ignore = io.gt_ignore;
    P.acc = w.acc; P.inst_area = io.inst_area; P.inst_inter = io.inst_inter;
    P.seg_prob_sum = io.seg_prob_sum; if (const BtIOSoftDice *sd = soft_io(p, io)) P.seg_soft2 = reinterpret_cast<long long *>(sd->seg_soft2);
    P.sweep = static_cast<long long *>(io.sweep); P.image_offset = p.image_offset; P.drop_gt_no_cand = p.drop_gt_no_cand; P.image_base = io.image_base;
    P.centre_cull = (p.iou_thres >= 0.55) ? 1 : 0;
    P.crop = p.crop; P.PW = p.proto_w; P.PH = p.proto_h;
    P.rx = (float)((double)p.proto_w / (double)p.img_w);
    P.ry = (float)((double)p.proto_h / (double)p.img_h);
    P.det_region = w.det_region;
    P.scr_off = w.scr_off; P.pool_used = w.pool_used; P.pool_cap = w.pool_cap;
    P.items = w.items; P.n_items = w.n_items; P.item_cap = (int)w.item_cap;
    P.tile_cnt = w.tile_cnt; P.tile_list = w.tile_list; P.ntiles = mask_tiles(&p); P.ntx = (p.proto_w + TA_W - 1) / TA_W;
    if (P.ntiles > PLAN_MAX_TILES) return BT_ERR_UNSUPPORTED;
    // centre-cell grid: cells of >= 64 px, at most 16 x 16
    P.gx = p.img_w / 64 < 1 ? 1 : (p.img_w / 64 > 16 ? 16 : p.img_w / 64);
    P.gy = p.img_h / 64 < 1 ? 1 : (p.img_h / 64 > 16 ? 16 : p.img_h / 64);
    P.inv_cw = (float)P.gx / (float)p.img_w;
    P.inv_ch = (float)P.gy / (float)p.img_h;

    // shared memory of nms_kernel: [sorted-index list | window (48 B/candidate) + kept arrays (48 B/slot)];
    // the sort's exchange buffer overlays everything.
    // BtParams.nms_threads = 512: 20 k registers (40 per thread) and 80 KB of shared memory per image leave room on the
    // SM for a second image and for CTAs of the other batches' kernels (btpost.Pipeline asks for it: 93.8 vs 98.7 us per
    // pipelined step, profiles/r02c_nms_threads.txt).  The 1024-thread variant (default) sorts lists of up to 16 384
    // candidates in shared memory; the small ones keep the pairs of lists above 4096 in the workspace.
    const int nt = p.nms_threads == 512 ? 512 : (p.nms_threads == 256 ? 256 : 1024);
    const int sort_max = nt <= 512 ? SORT_SMALL_MAX : SORT_REG_MAX;
    const int sort_slots = P.cap_pow2 < 1024 ? 1024 : (P.cap_pow2 > sort_max ? sort_max : P.cap_pow2);
    const size_t region0 = align_up((size_t)sort_slots * 4, 16);
    P.region0_bytes = (int)region0;
    size_t smem_a = region0 + (size_t)(nt == 512 ? NMS_WIN_512 : K2_TAIL_WIN) * 48 + (size_t)p.max_det * 48 + 64;
    if (smem_a < (size_t)sort_slots * 8) smem_a = (size_t)sort_slots * 8;
    {   // radix sort of short lists: two (key, index) buffers + [256][warps] counters
        const size_t mp = (size_t)(P.cap < RADIX_MAX ? (P.cap + 31) / 32 * 32 : RADIX_MAX);
        const size_t need = 16 * mp + 1024 * (size_t)(nt / 32);
        if (smem_a < need) smem_a = need;
    }
    {   // bucket rank sort: (key, index) pairs + two counter arrays behind region 0.  The 1024-thread variant owns its SM
        // anyway and grows its shared memory to take whole lists up to the register-sort limit; the smaller variants keep
        // their footprint (two images per SM) and take what fits.
        const size_t cap32 = (size_t)(P.cap + 31) / 32 * 32, fixed = region0 + 8 * (size_t)BUCKETS + 64;
        size_t want = cap32 < (size_t)sort_slots ? cap32 : (size_t)sort_slots;
        if (nt == 1024) {
            while (want > 0 && fixed + 8 * want > 200 * 1024) want -= 32;
            if (smem_a < fixed + 8 * want) smem_a = fixed + 8 * want;
        } else {
            while (want > 0 && fixed + 8 * want > smem_a) want -= 32;
        }
        P.bucket_max = (int)want;
        P.sort_stride = sort_stride_u64((size_t)P.cap);
    }
    // dynamic + static (~7 KB) shared memory of nms_kernel must stay below the 227 KB an SM offers one CTA: with 220 KB
    // the attribute call below was within 80 bytes of failing
    constexpr size_t NMS_SMEM_MAX = 212 * 1024;
    if (smem_a > NMS_SMEM_MAX) return BT_ERR_UNSUPPORTED;
    // match_kernel: COCO tables
    const int coco_doubles = p.max_det * 4 + p.max_gt * 4 + p.max_det * 4;   // boxes + room for a [K x 4] IoU block
    P.coco_smem_doubles = coco_doubles;
    const size_t smem_b = (size_t)coco_doubles * 8 + (size_t)p.max_det * 12 + 8 + (size_t)p.max_det * 16;   // + match-bit tables
    if (smem_b > 220 * 1024) return BT_ERR_UNSUPPORTED;
    // function attributes are per device: one flag per device ordinal
    static bool attr_done[64] = {};
    int attr_dev = 0;
    if (cudaGetDevice(&attr_dev) != cudaSuccess || attr_dev < 0 || attr_dev >= 64) return BT_ERR_CUDA;
    if (!attr_done[attr_dev]) {
        if (cudaFuncSetAttribute(nms_kernel<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NMS_SMEM_MAX) != cudaSuccess ||
            cudaFuncSetAttribute(nms_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NMS_SMEM_MAX) != cudaSuccess ||
            cudaFuncSetAttribute(nms_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NMS_SMEM_MAX) != cudaSuccess ||
            cudaFuncSetAttribute(match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess)
            return BT_ERR_CUDA;
        attr_done[attr_dev] = true;
    }
    if (parts & BT_NMS_SORT_SWEEP) {
        // measured and not kept: the highest launch priority for this kernel (the long pole of a step; it needs whole
        // SMs): one batch in flight 205.6 -> 198.5 us, but four in flight 539 k -> 524 k images/s
        if (nt == 256) nms_kernel<256><<<p.batch, nt, smem_a, s>>>(P);
        else if (nt == 512) nms_kernel<512><<<p.batch, nt, smem_a, s>>>(P);
        else nms_kernel<1024><<<p.batch, nt, smem_a, s>>>(P);
        if (cudaGetLastError() != cudaSuccess) return BT_ERR_CUDA;
    }
    if (parts & BT_NMS_GATHER) coeff_gather_kernel<<<dim3((p.max_det + 7) / 8, p.batch), GM_THREADS, 0, s>>>(P);
    if (parts & BT_NMS_PLAN) plan_kernel<<<p.batch, GM_THREADS, 0, s>>>(P);
    if ((parts & BT_NMS_COCO) && io.dt_match) match_kernel<<<p.batch, GM_THREADS, smem_b, s>>>(P);
    return cudaGetLastError() == cudaSuccess ? BT_OK : BT_ERR_CUDA;
}

}  // namespace bt
