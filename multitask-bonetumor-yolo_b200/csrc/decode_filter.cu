// Kernel 1: fused box decode + class max/argmax + strict confidence filter + clamp + ORDERED
// stream compaction, with GT preparation and the anchor<->GT confusion-matrix matching riding on
// the same pass over the head tensor.
//
// Reference statements replaced (paths under /root/reference/src):
//   decode      running_main_v2.py:743-775 (L1) / Ultralytics xywh->xyxy on segment_preds_cat (L2,
//               main_modelv2.py:367-375)
//   filter      running_main_v2.py:788-795   (max over classes, > CONF_TH strict, clamp_ after gather)
//   GT prep     running_main_v2.py:842-882 (clamped mAP copy) and :403-433 (unclamped loss copy)
//   CM match    running_main_v2.py:435-449,476-486 + batch_bbox_iou :68-94
//
// B200 mapping: one thread-block CLUSTER of 8 CTAs per image (grid 8 x B).  Each CTA owns a
// contiguous eighth of the anchors, reads the 4+nc box/score rows with 16-byte vector loads
// (coalesced: the head is [C, N] row-major per image), counts its survivors, and the eight counts
// are exchanged through distributed shared memory so that every CTA knows its output offset
// without a second kernel, global atomics or spin-waits.  The candidate list therefore comes out
// in anchor order, which is what makes NMS keep indices comparable with the reference's.
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace bt {

constexpr int K1_MAX_THREADS = 1024;   // block size is chosen per launch so that one pass covers the CTA's anchors
constexpr int K1_MAX_WARPS = K1_MAX_THREADS / 32;
constexpr int K1_CLUSTER = 8;
constexpr int K1_MAX_GT = 32;

struct K1Params {
    const void *head;    // L2 (fp32 or bf16)
    const void *maps[3];   // L1 (fp32 or bf16)
    int lvl_off[4];      // anchor offset of each level (L1)
    int lvl_w[3];
    float lvl_stride[3];
    int reg_max;
    int N, nc, nm, C;    // C = rows per image in the head (4+nc+nm) / channels of a map (L1)
    float conf;
    int clamp;
    float img_w, img_h;
    int cap;
    const float *gt_rows;
    int n_rows, gt_mode, max_gt;
    float cm_thr;
    float4 *cand_box;
    float *cand_score;
    int32_t *cand_label, *cand_anchor, *n_cand;
    int32_t *gt_count, *gt_rows_total;
    float *gt_boxes, *gt_boxes_raw;
    int32_t *gt_labels;
    unsigned long long *cm;
    int32_t *cm_pos;
};

// Exclusive prefix of `c` over the block in thread order; `total` = block sum.  SHFL: the second level (<= 32 warp totals)
// is a shuffle scan done by every warp (L2 decoder); otherwise every thread walks the totals in shared memory (the L1
// decoder is short of registers: the shuffle version spilled more and cost 30 us on the 64 x 640^2 batch).
template <bool SHFL>
__device__ __forceinline__ int block_excl_scan(int c, int &total, int *s_warp) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    const int nw = (blockDim.x + 31) >> 5;
    int off = 0, tot = 0;
    if (SHFL) {
        const int wv = lane < nw ? s_warp[lane] : 0;
        int winc = wv;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int v = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += v;
        }
        off = __shfl_sync(0xffffffffu, winc - wv, wid);
        tot = __shfl_sync(0xffffffffu, winc, 31);
    } else {
        for (int w = 0; w < nw; ++w) {
            int v = s_warp[w];
            if (w < wid) off += v;
            tot += v;
        }
    }
    __syncthreads();
    total = tot;
    return off + incl - c;
}

struct Decoded {
    float x1, y1, x2, y2;  // raw (unclamped) xyxy
    float score;
    int label;
};

// ---- L2 decoder: rows 0..3 = cx, cy, w, h in pixels; rows 4..4+nc = class scores.
// BF16: the head arrives as bfloat16 (the reference validates under bf16-mixed and upcasts with .float()); every
// value is widened exactly (a 16-bit shift), so the results equal the fp32 path's on the upcast tensor.
template <int VEC, bool BF16 = false>
struct L2Decoder {
    const void *img;  // head + b*C*N (fp32 or bf16 elements)
    int N, nc;
    __device__ __forceinline__ void load_row(int row, int n, float (&v)[VEC]) const {
        if (BF16) {
            const unsigned short *p = static_cast<const unsigned short *>(img) + (size_t)row * N + n;
            if (VEC == 4) {
                const uint2 t = __ldg(reinterpret_cast<const uint2 *>(p));
                v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xffff0000u);
                v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xffff0000u);
            } else {
                v[0] = __uint_as_float((unsigned)__ldg(p) << 16);
            }
            return;
        }
        const float *p = static_cast<const float *>(img) + (size_t)row * N + n;
        if (VEC == 4) {
            float4 t = __ldg(reinterpret_cast<const float4 *>(p));
            v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        } else {
            v[0] = __ldg(p);
        }
    }
    __device__ __forceinline__ void scores(int n, float (&best)[VEC], int (&lab)[VEC]) const {
        load_row(4, n, best);
#pragma unroll
        for (int i = 0; i < VEC; ++i) lab[i] = 0;
        for (int c = 1; c < nc; ++c) {
            float s[VEC];
            load_row(4 + c, n, s);
#pragma unroll
            for (int i = 0; i < VEC; ++i)
                if (s[i] > best[i] || (s[i] != s[i] && best[i] == best[i])) { best[i] = s[i]; lab[i] = c; }   // torch .max: NaN is the maximum, first NaN wins
        }
    }
    __device__ __forceinline__ void boxes(int n, float (&x1)[VEC], float (&y1)[VEC], float (&x2)[VEC],
                                          float (&y2)[VEC]) const {
        float cx[VEC], cy[VEC], w[VEC], h[VEC];
        load_row(0, n, cx); load_row(1, n, cy); load_row(2, n, w); load_row(3, n, h);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            float hw = __fmul_rn(w[i], 0.5f), hh = __fmul_rn(h[i], 0.5f);
            x1[i] = __fsub_rn(cx[i], hw); y1[i] = __fsub_rn(cy[i], hh);
            x2[i] = __fadd_rn(cx[i], hw); y2[i] = __fadd_rn(cy[i], hh);
        }
    }
};

// ---- L1 decoder: three raw maps [4*R+nc, H, W]; DFL softmax expectation, anchors (x+.5,y+.5),
// stride = img/W, class score = sigmoid(logit)  (running_main_v2.py:743-775, dist2bbox :97-107).
template <bool BF16>
struct L1DecoderBase {
    const void *map[3];  // already offset to image b (fp32 or bf16 elements; bf16 is widened exactly, = .float())
    int off[4], w[3];
    float stride[3];
    int R, nc, N;
    __device__ __forceinline__ float ld(int l, size_t i) const {
        if (BF16) return __uint_as_float((unsigned)__ldg(static_cast<const unsigned short *>(map[l]) + i) << 16);
        return __ldg(static_cast<const float *>(map[l]) + i);
    }
    __device__ __forceinline__ int level(int n) const { return n >= off[2] ? 2 : (n >= off[1] ? 1 : 0); }
    __device__ __forceinline__ void scores1(int n, float (&best)[1], int (&lab)[1]) const {
        int l = level(n);
        int HW = off[l + 1] - off[l], pos = n - off[l];
        const size_t p = (size_t)(4 * R) * HW + pos;
        float b = -1.0f; int bi = 0;
        for (int c = 0; c < nc; ++c) {
            float lg = ld(l, p + (size_t)c * HW);
            float s = __fdiv_rn(1.0f, __fadd_rn(1.0f, bt_expf(-lg)));
            if (c == 0 || s > b || (s != s && b == b)) { b = s; bi = c; }   // torch .max: NaN is the maximum, first NaN wins
        }
        best[0] = b; lab[0] = bi;
    }
    __device__ __forceinline__ void boxes1(int n, float (&x1)[1], float (&y1)[1], float (&x2)[1], float (&y2)[1]) const {
        int l = level(n);
        int HW = off[l + 1] - off[l], pos = n - off[l];
        int W = w[l];
        int y = pos / W, x = pos - y * W;
        float st = stride[l];
        float d[4];
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const size_t p = (size_t)(s * R) * HW + pos;
            float m = ld(l, p);
            for (int k = 1; k < R; ++k) { float v = ld(l, p + (size_t)k * HW); if (v > m) m = v; }
            float sum = 0.0f, acc = 0.0f;
            for (int k = 0; k < R; ++k) {
                float e = bt_expf(__fsub_rn(ld(l, p + (size_t)k * HW), m));
                sum = __fadd_rn(sum, e);
                acc = __fmaf_rn(e, (float)k, acc);
            }
            d[s] = __fdiv_rn(acc, sum);
        }
        float ax = __fmul_rn(__fadd_rn((float)x, 0.5f), st), ay = __fmul_rn(__fadd_rn((float)y, 0.5f), st);
        x1[0] = __fsub_rn(ax, __fmul_rn(d[0], st));
        y1[0] = __fsub_rn(ay, __fmul_rn(d[1], st));
        x2[0] = __fadd_rn(ax, __fmul_rn(d[2], st));
        y2[0] = __fadd_rn(ay, __fmul_rn(d[3], st));
    }
};

template <int VEC, bool BF16>
struct L1Decoder : L1DecoderBase<BF16> {
    using Base = L1DecoderBase<BF16>;
    int astep;    // distance between the VEC anchors of a thread (interleaved mapping: consecutive lanes = consecutive anchors)
    __device__ __forceinline__ void scores(int n, float (&best)[VEC], int (&lab)[VEC]) const {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            float b1[1] = {0.0f}; int l1[1] = {0};
            if (n + i * astep < Base::N) Base::scores1(n + i * astep, b1, l1);
            best[i] = b1[0]; lab[i] = l1[0];
        }
    }
    __device__ __forceinline__ void boxes(int n, float (&x1)[VEC], float (&y1)[VEC], float (&x2)[VEC], float (&y2)[VEC]) const {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            float a[1] = {0.0f}, b[1] = {0.0f}, c[1] = {0.0f}, d[1] = {0.0f};
            if (n + i * astep < Base::N) Base::boxes1(n + i * astep, a, b, c, d);
            x1[i] = a[0]; y1[i] = b[0]; x2[i] = c[0]; y2[i] = d[0];
        }
    }
};

// INTERLEAVED: thread t of the CTA owns anchors a0 + t, a0 + cnt + t, ... (cnt = anchors per pass) instead of VEC
// consecutive ones: for the channel-planar raw maps (L1) every load of a warp is then one contiguous line, and the
// ordered compaction runs one block scan per pass.
template <int VEC, bool INTERLEAVED, class Dec>
__device__ __forceinline__ void k1_body(const K1Params &P, Dec &dec, int b) {
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int tid = threadIdx.x, lane = tid & 31;

    __shared__ int s_warp[K1_MAX_WARPS];
    __shared__ int s_ex;                 // this CTA's survivor count, read by peers through DSMEM
    __shared__ float s_coord[K1_MAX_GT][4];
    __shared__ __align__(16) float s_gtraw[K1_MAX_GT * 4];
    __shared__ int s_gl[K1_MAX_GT];
    __shared__ int s_G;
    __shared__ int s_cm[BT_MAX_CLASSES * BT_MAX_CLASSES];
    __shared__ int s_npos;

    for (int i = tid; i < BT_MAX_CLASSES * BT_MAX_CLASSES; i += blockDim.x) s_cm[i] = 0;
    if (tid == 0) s_npos = 0;

    // ---- anchor range of this CTA (in groups of VEC anchors); the block is sized so that every
    // group has its own thread: ONE pass, the decoded values stay in registers across the
    // cluster exchange (ncu r01b: the two-pass / two-iteration version spent its time in barriers
    // waiting for a second round of loads that only 7 threads needed).
    const int groups = (P.N + VEC - 1) / VEC;
    const int gp = (groups + K1_CLUSTER - 1) / K1_CLUSTER;
    const int g0 = rank * gp, g1 = min(groups, g0 + gp);
    const int nthreads = blockDim.x;

    // issue the head loads first: they are in flight while the GT rows are gathered
    float best[VEC], x1[VEC], y1[VEC], x2[VEC], y2[VEC];
    int lab[VEC];
    const int g = g0 + tid;
    const bool active = g < g1;
    const int cnt = g1 - g0;                                     // threads in use = anchors per pass
    auto anchor_of = [&](int i) { return INTERLEAVED ? g0 * VEC + i * cnt + tid : g * VEC + i; };
    if (active) {
        dec.scores(anchor_of(0), best, lab);
        dec.boxes(anchor_of(0), x1, y1, x2, y2);
    }

    // ---- GT prep: ordered gather of this image's rows, then the reference's cat/view layout.
    {
        const float S = P.img_w;  // reference multiplies every coordinate by the scalar img_size
        int base = 0;
        for (int r0 = 0; r0 < P.n_rows; r0 += nthreads) {
            int r = r0 + tid;
            bool hit = false;
            float row[6];
            if (r < P.n_rows) {
#pragma unroll
                for (int k = 0; k < 6; ++k) row[k] = __ldg(P.gt_rows + (size_t)r * 6 + k);
                hit = (row[0] == (float)b);
            }
            int tot;
            int pos = base + block_excl_scan<!INTERLEAVED>(hit ? 1 : 0, tot, s_warp);
            if (hit && pos < P.max_gt) {
                float cx = row[2], cy = row[3], w = row[4], h = row[5];
                float hw = __fdiv_rn(w, 2.0f), hh = __fdiv_rn(h, 2.0f);
                s_coord[pos][0] = __fmul_rn(__fsub_rn(cx, hw), S);
                s_coord[pos][1] = __fmul_rn(__fsub_rn(cy, hh), S);
                s_coord[pos][2] = __fmul_rn(__fadd_rn(cx, hw), S);
                s_coord[pos][3] = __fmul_rn(__fadd_rn(cy, hh), S);
                s_gl[pos] = (int)row[1];
            }
            base += tot;
        }
        if (tid == 0) s_G = base < P.max_gt ? base : P.max_gt;
        __syncthreads();
        const int G = s_G;
        for (int i = tid; i < 4 * G; i += nthreads) {
            float v = (P.gt_mode == BT_GT_LITERAL) ? s_coord[i % G][i / G] : s_coord[i / 4][i % 4];
            s_gtraw[i] = v;
            if (rank == 0) {
                P.gt_boxes_raw[(size_t)b * P.max_gt * 4 + i] = v;
                P.gt_boxes[(size_t)b * P.max_gt * 4 + i] = fminf(fmaxf(v, 0.0f), S);
            }
        }
        if (rank == 0) {
            // padding beyond the image's boxes is zero-filled: the outputs do not depend on what a previous batch left
            for (int i = 4 * G + tid; i < 4 * P.max_gt; i += nthreads) {
                P.gt_boxes_raw[(size_t)b * P.max_gt * 4 + i] = 0.0f;
                P.gt_boxes[(size_t)b * P.max_gt * 4 + i] = 0.0f;
            }
            for (int i = G + tid; i < P.max_gt; i += nthreads) P.gt_labels[(size_t)b * P.max_gt + i] = 0;
            for (int i = tid; i < G; i += nthreads) P.gt_labels[(size_t)b * P.max_gt + i] = s_gl[i];
            if (tid == 0) {
                P.gt_count[b] = G;
                if (P.gt_rows_total) P.gt_rows_total[b] = base;   // before the max_gt cut: the host raises when it is larger
            }
        }
        __syncthreads();
    }
    const int G = s_G;

    // ---- filter flags + anchor<->GT confusion-matrix matching on the raw boxes
    int c = 0, npos_thread = 0;
    unsigned flags = 0;
    if (active) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            if (anchor_of(i) >= P.N) continue;
            if (best[i] > P.conf) { flags |= 1u << i; ++c; }
            if (G > 0) {
                // batch_bbox_iou (running_main_v2.py:68-94) against the unclamped GT copy.  With a
                // non-negative threshold an anchor that intersects no GT box can never be positive
                // (every IoU is 0/x), so the divisions are skipped for it; otherwise the full
                // max / first-argmax over GT is evaluated exactly as the reference does.
                bool any = P.cm_thr < 0.0f;
                for (int q = 0; q < G && !any; ++q) {
                    const float4 gq = reinterpret_cast<const float4 *>(s_gtraw)[q];
                    float iw = __fsub_rn(fminf(x2[i], gq.z), fmaxf(x1[i], gq.x));
                    float ih = __fsub_rn(fminf(y2[i], gq.w), fmaxf(y1[i], gq.y));
                    any = (iw > 0.0f) && (ih > 0.0f);
                }
                if (!any) continue;
                float a1 = __fmul_rn(__fsub_rn(x2[i], x1[i]), __fsub_rn(y2[i], y1[i]));
                float bi = 0.0f; int bg = 0;
                for (int q = 0; q < G; ++q) {
                    const float4 gq = reinterpret_cast<const float4 *>(s_gtraw)[q];
                    float qx1 = gq.x, qy1 = gq.y, qx2 = gq.z, qy2 = gq.w;
                    float ix1 = fmaxf(x1[i], qx1), iy1 = fmaxf(y1[i], qy1);
                    float ix2 = fminf(x2[i], qx2), iy2 = fminf(y2[i], qy2);
                    float iw = __fsub_rn(ix2, ix1); iw = iw < 0.0f ? 0.0f : iw;
                    float ih = __fsub_rn(iy2, iy1); ih = ih < 0.0f ? 0.0f : ih;
                    float inter = __fmul_rn(iw, ih);
                    float a2 = __fmul_rn(__fsub_rn(qx2, qx1), __fsub_rn(qy2, qy1));
                    float uni = __fsub_rn(__fadd_rn(a1, a2), inter);
                    float iou = __fdiv_rn(inter, __fadd_rn(uni, 1e-7f));
                    if (q == 0 || iou > bi) { bi = iou; bg = q; }
                }
                if (bi > P.cm_thr) {
                    int gc = s_gl[bg], pc = lab[i];
                    if (gc >= 0 && gc < P.nc && pc >= 0 && pc < P.nc) atomicAdd(&s_cm[gc * P.nc + pc], 1);
                    ++npos_thread;
                }
            }
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) npos_thread += __shfl_down_sync(0xffffffffu, npos_thread, d);
    if (lane == 0 && npos_thread) atomicAdd(&s_npos, npos_thread);
    // ---- ordered offsets: block scan, then the eight CTA totals through distributed shared memory
    int my_total, excl = 0, exclv[VEC];
    if (INTERLEAVED) {
        int run = 0;
#pragma unroll
        for (int i = 0; i < VEC; ++i) {   // anchor order = pass-major
            int tot;
            exclv[i] = run + block_excl_scan<false>((flags >> i) & 1u, tot, s_warp);
            run += tot;
        }
        my_total = run;
    } else {
        excl = block_excl_scan<true>(c, my_total, s_warp);
    }
    if (tid == 0) s_ex = my_total;
    cluster.sync();
    int base = 0, all = 0;
    for (int r = 0; r < K1_CLUSTER; ++r) {
        int v = *cluster.map_shared_rank(&s_ex, r);
        if (r < rank) base += v;
        all += v;
    }
    if (rank == 0 && tid == 0) P.n_cand[b] = all < P.cap ? all : P.cap;
    // confusion-matrix counts: rank 0 folds the eight CTAs' shared-memory histograms (DSMEM reads)
    // and issues ONE global atomic per non-zero cell and image (512 CTAs hammering the same nine
    // addresses serialised in L2 and dominated the first version of this kernel).
    if (rank == 0) {
        for (int i = tid; i < P.nc * P.nc; i += nthreads) {
            int v = 0;
            for (int r = 0; r < K1_CLUSTER; ++r) v += cluster.map_shared_rank(s_cm, r)[i];
            if (v) atomicAdd(&P.cm[i], (unsigned long long)v);
        }
        if (tid == 0) {
            int v = 0;
            for (int r = 0; r < K1_CLUSTER; ++r) v += *cluster.map_shared_rank(&s_npos, r);
            P.cm_pos[b] = v;
        }
    }
    if (flags) {
        int pos = base + excl;
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            if (!(flags & (1u << i))) continue;
            if (INTERLEAVED) pos = base + exclv[i];
            if (pos < P.cap) {
                float bx1 = x1[i], by1 = y1[i], bx2 = x2[i], by2 = y2[i];
                if (P.clamp) {
                    bx1 = fminf(fmaxf(bx1, 0.0f), P.img_w); bx2 = fminf(fmaxf(bx2, 0.0f), P.img_w);
                    by1 = fminf(fmaxf(by1, 0.0f), P.img_h); by2 = fminf(fmaxf(by2, 0.0f), P.img_h);
                }
                size_t o = (size_t)b * P.cap + pos;
                P.cand_box[o] = make_float4(bx1, by1, bx2, by2);
                P.cand_score[o] = best[i];
                P.cand_label[o] = lab[i];
                P.cand_anchor[o] = anchor_of(i);
            }
            ++pos;
        }
    }
    cluster.sync();  // peers may still be reading s_ex / s_cm through DSMEM
}

// MAXT = 320: blocks of <= 320 threads, at least 4 resident per SM so that the 8 x B CTAs of a
// 64-image batch form a single wave (ncu r01c: 64 registers -> 3 CTAs/SM -> a second wave doubled
// the kernel time).  MAXT = 1024: large anchor counts.
template <int VEC, int MAXT, bool BF16 = false>
__global__ void __cluster_dims__(K1_CLUSTER, 1, 1) __launch_bounds__(MAXT, MAXT <= 320 ? 4 : 1)
decode_filter_l2_kernel(const __grid_constant__ K1Params P) {
    const int b = blockIdx.y;
    L2Decoder<VEC, BF16> dec{static_cast<const char *>(P.head) + (size_t)b * P.C * P.N * (BF16 ? 2 : 4), P.N, P.nc};
    k1_body<VEC, false>(P, dec, b);
}

// MAXT = 320: four anchors per thread in blocks small enough for 4 CTAs per SM, so the whole batch is one wave
// and the DFL arithmetic (64 exp per anchor) has ~36 warps per SM to hide behind (r02: one anchor per thread in
// 1056-thread blocks ran at 1 CTA per SM in 3.5 waves, 180 us).
template <int VEC, int MAXT, bool BF16 = false>
__global__ void __cluster_dims__(K1_CLUSTER, 1, 1) __launch_bounds__(MAXT, MAXT <= 320 ? 4 : 1)
decode_filter_l1_kernel(const __grid_constant__ K1Params P) {
    const int b = blockIdx.y;
    L1Decoder<VEC, BF16> dec;
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        int HW = P.lvl_off[l + 1] - P.lvl_off[l];
        dec.map[l] = static_cast<const char *>(P.maps[l]) + (size_t)b * P.C * HW * (BF16 ? 2 : 4);
        dec.off[l] = P.lvl_off[l];
        dec.w[l] = P.lvl_w[l];
        dec.stride[l] = P.lvl_stride[l];
    }
    dec.off[3] = P.lvl_off[3];
    dec.R = P.reg_max;
    dec.nc = P.nc;
    dec.N = P.N;
    {
        // anchors per pass of this CTA (same expression as in k1_body)
        const int groups = (P.N + VEC - 1) / VEC, gp = (groups + K1_CLUSTER - 1) / K1_CLUSTER;
        const int r = (int)cg::this_cluster().block_rank();
        dec.astep = min(groups, r * gp + gp) - r * gp;
    }
    k1_body<VEC, true>(P, dec, b);
}

int launch_decode_filter(const BtParams &p, const BtIO &io, const Workspace &w, cudaStream_t s) {
    K1Params P{};
    P.N = p.num_anchors; P.nc = p.nc; P.nm = p.nm;
    P.conf = p.conf_thres; P.clamp = p.clamp_boxes;
    P.img_w = (float)p.img_w; P.img_h = (float)p.img_h;
    P.cap = cand_capacity(&p);
    P.gt_rows = io.det_boxes_gt; P.n_rows = io.det_boxes_gt ? p.num_gt_rows : 0;
    P.gt_mode = p.gt_mode; P.max_gt = p.max_gt; P.cm_thr = p.iou_match_thresh;
    P.cand_box = w.cand_box; P.cand_score = w.cand_score; P.cand_label = w.cand_label;
    P.cand_anchor = w.cand_anchor; P.n_cand = io.n_cand;
    P.gt_count = io.gt_count; P.gt_rows_total = io.gt_rows_total; P.gt_boxes = io.gt_boxes; P.gt_boxes_raw = io.gt_boxes_raw;
    P.gt_labels = io.gt_labels;
    P.cm = reinterpret_cast<unsigned long long *>(io.cm); P.cm_pos = io.cm_pos;
    auto block_for = [&](int vecw) {
        int groups = (p.num_anchors + vecw - 1) / vecw;
        int gp = (groups + K1_CLUSTER - 1) / K1_CLUSTER;
        return (gp + 31) / 32 * 32;
    };
    dim3 grid(K1_CLUSTER, p.batch);
    if (p.layout == BT_LAYOUT_L2) {
        P.head = io.head; P.C = 4 + p.nc + p.nm;
        const bool bf16 = p.head_dtype == BT_HEAD_BF16;
        bool vec = (p.num_anchors % 4 == 0) && ((reinterpret_cast<uintptr_t>(io.head) & 15) == 0);
        if (block_for(vec ? 4 : 1) > K1_MAX_THREADS) return BT_ERR_UNSUPPORTED;  // > 32768 (262144 vectorised) anchors
        dim3 block(block_for(vec ? 4 : 1));
        const bool small = block.x <= 320;
        if (bf16) {
            if (vec && small) decode_filter_l2_kernel<4, 320, true><<<grid, block, 0, s>>>(P);
            else if (vec) decode_filter_l2_kernel<4, 1024, true><<<grid, block, 0, s>>>(P);
            else if (small) decode_filter_l2_kernel<1, 320, true><<<grid, block, 0, s>>>(P);
            else decode_filter_l2_kernel<1, 1024, true><<<grid, block, 0, s>>>(P);
        } else if (vec && block.x <= 288) decode_filter_l2_kernel<4, 288><<<grid, block, 0, s>>>(P);   // 8400 anchors: 56 registers, no second wave
        else if (vec && small) decode_filter_l2_kernel<4, 320><<<grid, block, 0, s>>>(P);
        else if (vec) decode_filter_l2_kernel<4, 1024><<<grid, block, 0, s>>>(P);
        else if (small) decode_filter_l2_kernel<1, 320><<<grid, block, 0, s>>>(P);
        else decode_filter_l2_kernel<1, 1024><<<grid, block, 0, s>>>(P);
    } else {
        P.C = 4 * p.reg_max + p.nc; P.reg_max = p.reg_max;
        int off = 0;
        const int strides[3] = {8, 16, 32};
        for (int l = 0; l < 3; ++l) {
            int W = p.img_w / strides[l], H = p.img_h / strides[l];
            P.maps[l] = io.maps[l];
            P.lvl_off[l] = off; P.lvl_w[l] = W;
            P.lvl_stride[l] = (float)p.img_w / (float)W;  // running_main_v2.py:726
            off += W * H;
        }
        P.lvl_off[3] = off;
        const bool bf16 = p.head_dtype == BT_HEAD_BF16;   // raw maps of a bf16-mixed forward (running_main_v2.py:1324)
        if (bf16) {
            if (block_for(4) <= 320) decode_filter_l1_kernel<4, 320, true><<<grid, dim3(block_for(4)), 0, s>>>(P);
            else if (block_for(1) <= K1_MAX_THREADS) decode_filter_l1_kernel<1, K1_MAX_THREADS, true><<<grid, dim3(block_for(1)), 0, s>>>(P);
            else if (block_for(2) <= K1_MAX_THREADS) decode_filter_l1_kernel<2, K1_MAX_THREADS, true><<<grid, dim3(block_for(2)), 0, s>>>(P);
            else if (block_for(4) <= K1_MAX_THREADS) decode_filter_l1_kernel<4, K1_MAX_THREADS, true><<<grid, dim3(block_for(4)), 0, s>>>(P);
            else return BT_ERR_UNSUPPORTED;
        } else if (block_for(4) <= 320) decode_filter_l1_kernel<4, 320><<<grid, dim3(block_for(4)), 0, s>>>(P);
        else if (block_for(1) <= K1_MAX_THREADS) decode_filter_l1_kernel<1, K1_MAX_THREADS><<<grid, dim3(block_for(1)), 0, s>>>(P);
        else if (block_for(2) <= K1_MAX_THREADS) decode_filter_l1_kernel<2, K1_MAX_THREADS><<<grid, dim3(block_for(2)), 0, s>>>(P);
        else if (block_for(4) <= K1_MAX_THREADS) decode_filter_l1_kernel<4, K1_MAX_THREADS><<<grid, dim3(block_for(4)), 0, s>>>(P);
        else return BT_ERR_UNSUPPORTED;
    }
    return cudaGetLastError() == cudaSuccess ? BT_OK : BT_ERR_CUDA;
}

}  // namespace bt
