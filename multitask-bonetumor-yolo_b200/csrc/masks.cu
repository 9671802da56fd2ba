// Stage 3: mask assembly + segmentation counters.
//
// Reference statements replaced (paths under /root/reference/src):
//   M1 projector   running_main_v2.py:689-703 (Conv2d(32->1,k=1) -> F.interpolate bilinear x4,
//                  align_corners=False -> sigmoid -> >0.5 -> int), evaluate_model.py:160-171
//   M2 instance    test_model.py:80-85 (einsum coeff x protos -> bilinear -> sigmoid>0.5) with the
//                  Ultralytics process_mask crop at prototype resolution (SURVEY.md A.5)
//   counters       running_main_v2.py:704-713 (tp/fp/fn/tn, DiceScore) and test_model.py:15-23
//                  (per-image IoU / Dice with eps 1e-7)
//
// B200 mapping: four kernels, each bound by one resource (plan_kernel in nms_match.cu prepares their work lists).
//   gt_pack_kernel    GT mask bytes -> bits, one 64-bit word per 2x2 block of cells (a cell = the 4x4
//                     output pixels between four neighbouring prototype pixels).  Pure streaming; independent of
//                     the detections, so btpost_run runs it on its helper stream beside decode / NMS.
//   contract_kernel   THE pass over the prototypes (2/3 of the path's compulsory HBM bytes): persistent CTAs, 4 per
//                     SM, each a contiguous range of 32 x 8 pixel tiles; a tile of all 32 channels arrives with ONE
//                     3-D tensor-map TMA (128-byte swizzle; bf16 prototypes: 64-byte swizzle) with an L2 evict-first
//                     hint, every thread moves its two pixels x 32 channels into registers, the buffer is re-armed
//                     for the next tile at once, and the K=32 contraction of the projector and of every detection
//                     the plan binned into the tile is 32 packed FFMA2 per (detection, pixel pair) with the
//                     coefficients broadcast from shared memory: no prototype re-reads, no search, sequential fp32
//                     order (bit parity with torch).  Logits go to an L2-resident scratch (projector: [B,PH,PW];
//                     detections: their crop boxes back to back in a pool).  HBM-bound (75 % of the measured peak).
//   cells_kernel      bilinear x4 + threshold on 2x2 cell blocks: 9 corner logits -> 64 output pixels with
//                     packed FMUL2/FFMA2 (two pixels per instruction), the threshold as the sign bit of a
//                     packed subtraction gathered by one funnel shift per pixel.  Persistent warps pull (detection,
//                     chunk of 128 blocks) items and runs of 32 projector blocks off 32 queue counters; the union of
//                     an image's instance masks is a 64-bit atomic OR per block whose returned old word gives the
//                     newly set bits (union counters without a pass over the union); the projector mask owns its
//                     cells.  Instruction-issue bound.
//   finalize_kernel   one warp per image: counters -> Dice / IoU / tp-fp-fn-tn, the image's v3 segmentation-mAP
//                     record when BtIO.seg_sweep is set, and its v3 soft Dice when BtIOSoftDice.seg_soft2 is set.
// A fifth kernel, seg_curve_kernel (btpost_seg_curve, its own entry point), runs after them when the caller asks for the
// binned PR / ROC state of the projector probabilities.
// tcgen05 is deliberately not used: K = 32 at <= 0.5 FLOP/B, and TF32/BF16 accumulation would break the bit
// parity of the thresholded masks with the fp32 reference.
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"

namespace bt {

constexpr int NM = 32;
constexpr int A_THREADS = 128;          // 4 warps, each an 8 x 8 pixel block, 2 pixels per thread
constexpr int A_LCAP = 32;              // detections staged per round
constexpr int C_THREADS = 256;
constexpr int G_THREADS = 128, G_ROWS = 4;   // gt_pack_kernel: threads, rows of blocks per CTA
constexpr int C_NQ = 32, C_QSTRIDE = 32;   // work queues of cells_kernel: counters 128 bytes apart

typedef unsigned long long u64;

struct K3Params {
    int B, S_h, S_w, PH, PW, K, gt_f32, proto_bf16, NBY, NBX, ntx, nty, m1_items, nq;
    float bias, inv_K;
    const int2 *items;      // plan of the cells kernel: (image * K + detection, chunk)
    const int32_t *n_items;
    float inv_m1;
    int item_cap;
    const void *protos;     // [B, NM, PH, PW] fp32 or bfloat16 (proto_bf16)
    const float *proj_weight, *det_coeff;
    const int32_t *det_count, *scr_off, *tile_cnt;
    const unsigned short *tile_list;
    const short4 *det_region;
    const void *masks_gt;
    float *pool, *lm;
    u64 *gtc, *unc;
    int32_t *gpart, *work, *acc, *inst_area, *inst_inter;
    long long *seg_cnt4, *uni_cnt4, *seg_img3, *uni_img3;
    float *seg_dice, *seg_iou, *uni_dice, *uni_iou;
    uint8_t *seg_mask, *uni_mask;
    uint32_t *inst_bits;    // [B, K, S_h, S_w / 32] optional: every instance mask, bit-packed (zeroed before cells_kernel)
    uint8_t *inst_masks;    // [B, K, S_h, S_w] optional: the same as bytes, expanded from inst_bits
    float *seg_logits;
    double *seg_prob_sum;   // [B] optional: sum of sigmoid(logit) over the projector mask's foreground pixels
    long long *sweep;       // optional sweep state: per-image Dice / IoU are added to its header (2^-40 fixed point)
    u64 valid_tab[9];       // valid-pixel mask of a block by (row class, column class): first / interior / last
    float inv_NBX;
    // v3 segmentation mAP (BtIO.seg_sweep); appended last so that the fields above keep their parameter offsets
    long long *seg_sweep;   // optional sweep state: one record per image, written by finalize_kernel
    const int32_t *image_base;
    int image_offset, T;
    double thrs[BT_MAX_IOU_THRS];
    // v3 soft Dice (BtIOSoftDice.seg_soft2 / seg_soft_dice / seg_soft_acc); appended last for the same reason
    long long *seg_soft2;   // [B, 2] optional: sum of p * t and of p, 2^-40 fixed point (zeroed by the NMS kernel)
    float *seg_soft_dice;
    long long *seg_soft_acc;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// One [NM][TA_H][TA_W] box of the [B*NM, PH, PW] prototype tensor -> shared memory.
// The prototypes are read exactly once: L2 evict-first keeps the logit pool, the projector logits and the GT / union
// words resident for cells_kernel instead of 210 MB of stream-through data.
__device__ __forceinline__ void tma_tile_g2s(void *dst, const CUtensorMap *tm, int col, int row, int chan0, uint64_t *bar,
                                             bool keep) {
    // keep: some detection has no room in the logit pool, cells_kernel will contract its corners from the prototypes
    uint64_t policy;
    if (keep) asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(policy));
    else asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(col), "r"(row), "r"(chan0), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(void *dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(void *dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}

// ---- packed fp32x2 arithmetic (sm_100: FFMA2 / FMUL2, one issue slot for two results; every lane rounds
// exactly like the scalar instruction)
__device__ __forceinline__ u64 pack2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(u64 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ void unpack2u(u64 v, uint32_t &lo, uint32_t &hi) { asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v)); }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
    u64 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
    u64 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// torch's bilinear kernel order, pinned in the oracle: fma(h0, fma(w0,v00,w1*v01), h1*fma(w0,v10,w1*v11))
__device__ __forceinline__ float lerp_row(float a, float b, float w0, float w1) {
    return __fmaf_rn(w0, a, __fmul_rn(w1, b));
}

// Scalar cell evaluation with the logits kept (dense-output / score paths only): 4 corner values -> 4x4
// thresholded output pixels, bit (ry*4+rx).  Border cells (index -1) use interpolation weight 0.
__device__ __forceinline__ unsigned cell_bits_log(float v00, float v01, float v10, float v11, bool border_y, bool border_x,
                                                  float (&logits)[16]) {
    float top[4], bot[4];
#pragma unroll
    for (int rx = 0; rx < 4; ++rx) {
        float w1 = border_x ? 0.0f : (0.125f + 0.25f * rx);
        float w0 = 1.0f - w1;
        top[rx] = lerp_row(v00, v01, w0, w1);
        bot[rx] = lerp_row(v10, v11, w0, w1);
    }
    unsigned bits = 0;
#pragma unroll
    for (int ry = 0; ry < 4; ++ry) {
        float h1 = border_y ? 0.0f : (0.125f + 0.25f * ry);
        float h0 = 1.0f - h1;
#pragma unroll
        for (int rx = 0; rx < 4; ++rx) {
            float v = __fmaf_rn(h0, top[rx], __fmul_rn(h1, bot[rx]));
            logits[ry * 4 + rx] = v;
            if (sigmoid_gt_half(v)) bits |= 1u << (ry * 4 + rx);
        }
    }
    return bits;
}

// Valid-pixel mask of a cell: border cells (-1) own output rows/cols {0,1}; the last cell row/col
// owns only the two pixels left before the image edge; cells past the last one do not exist.
__host__ __device__ __forceinline__ unsigned cell_valid(int ci, int cj, int PH, int PW, int S_h, int S_w) {
    if (ci > PH - 1 || cj > PW - 1) return 0u;
    const int nry = (ci < 0) ? 2 : (S_h - (4 * ci + 2) < 4 ? S_h - (4 * ci + 2) : 4);
    const int nrx = (cj < 0) ? 2 : (S_w - (4 * cj + 2) < 4 ? S_w - (4 * cj + 2) : 4);
    const unsigned rowm = (1u << nrx) - 1u;
    unsigned m = 0;
    for (int r = 0; r < nry; ++r) m |= rowm << (4 * r);
    return m;
}

// ---- 2x2 cell blocks.  Block (by, bx) holds the cells ci in {2by-1, 2by}, cj in {2bx-1, 2bx}; its 64-bit
// word is cell (a, c) at bits 16*(2a+c) .. +15, pixel (ry, rx) of a cell at bit 4*ry+rx.
struct BlockGeo {
    int r0, r1, r2, c0, c1, c2;   // prototype rows / columns of the 3x3 corner logits
};
__device__ __forceinline__ BlockGeo block_geo(int by, int bx, int PH, int PW) {
    BlockGeo g;
    // cell row A (ci = 2by-1) interpolates rows (r0, r1), cell row B (ci = 2by) rows (by ? r1 : r0, r2): the border
    // cell -1 reads the same rows (0, 1) as cell 0 with weight 0 on the second; past the last row the lower corner is
    // the upper one (source index clamped).  PH, PW >= 2.
    g.r0 = max(2 * by - 1, 0);
    g.r1 = max(min(2 * by, PH - 1), 1);
    g.r2 = min(2 * by + 1, PH - 1);
    g.c0 = max(2 * bx - 1, 0);
    g.c1 = max(min(2 * bx, PW - 1), 1);
    g.c2 = min(2 * bx + 1, PW - 1);
    return g;
}

// Valid-pixel mask of a block.  Only the first and the last block row / column differ from all-ones, so the host
// computes the nine masks once (`valid_tab`, launch_masks) and the kernels look them up.
__host__ __device__ __forceinline__ u64 block_valid_slow(int by, int bx, int PH, int PW, int S_h, int S_w) {
    const int ciA = 2 * by - 1, cjA = 2 * bx - 1;
    const u64 vAA = cell_valid(ciA, cjA, PH, PW, S_h, S_w), vAB = cell_valid(ciA, cjA + 1, PH, PW, S_h, S_w);
    const u64 vBA = cell_valid(ciA + 1, cjA, PH, PW, S_h, S_w), vBB = cell_valid(ciA + 1, cjA + 1, PH, PW, S_h, S_w);
    return vAA | (vAB << 16) | (vBA << 32) | (vBB << 48);
}
__device__ __forceinline__ u64 block_valid(const K3Params &P, int by, int bx) {
    if ((unsigned)(by - 1) < (unsigned)(P.NBY - 2) && (unsigned)(bx - 1) < (unsigned)(P.NBX - 2)) return ~0ull;   // interior: the common case
    const int rc = by == 0 ? 0 : (by == P.NBY - 1 ? 2 : 1), cc = bx == 0 ? 0 : (bx == P.NBX - 1 ? 2 : 1);
    return P.valid_tab[rc * 3 + cc];
}

// Thresholded pixels of a 2x2 cell block from its 3x3 corner logits v[row][col] (unmasked).  BY0 / BX0: the block
// holds the border cells of row / column -1 (compile-time: interior blocks carry no selects).
template <bool BY0, bool BX0>
__device__ __forceinline__ u64 block_bits_t(const float (&v)[3][3]) {
    // horizontal interpolation of the three rows for the two cell columns, two pixels per instruction
    const u64 W1a = pack2(0.125f, 0.375f), W1b = pack2(0.625f, 0.875f);
    const u64 W0a = pack2(0.875f, 0.625f), W0b = pack2(0.375f, 0.125f);
    const u64 ONE = pack2(1.0f, 1.0f), ZERO = pack2(0.0f, 0.0f);
    const u64 wA0a = BX0 ? ONE : W0a, wA0b = BX0 ? ONE : W0b, wA1a = BX0 ? ZERO : W1a, wA1b = BX0 ? ZERO : W1b;
    u64 hA[3][2], hB[3][2];   // [row][pixel pair] of cell column A / B
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float lA = v[i][0], rA = v[i][1];
        const float lB = BX0 ? v[i][0] : v[i][1], rB = v[i][2];
        const u64 lA2 = pack2(lA, lA), rA2 = pack2(rA, rA), lB2 = pack2(lB, lB), rB2 = pack2(rB, rB);
        hA[i][0] = fma2(wA0a, lA2, mul2(wA1a, rA2));
        hA[i][1] = fma2(wA0b, lA2, mul2(wA1b, rA2));
        hB[i][0] = fma2(W0a, lB2, mul2(W1a, rB2));
        hB[i][1] = fma2(W0b, lB2, mul2(W1b, rB2));
    }
    // sigmoid(x) > 0.5  <=>  x > T0  <=>  sign bit of (T0 - x); NaN gives the canonical positive NaN (false)
    const u64 T0 = pack2(8.940696716308594e-08f, 8.940696716308594e-08f), NEG1 = pack2(-1.0f, -1.0f);
    uint32_t word[2];
#pragma unroll
    for (int a = 0; a < 2; ++a) {          // cell row A / B
        const int it = (a == 1 && !BY0) ? 1 : 0;   // top row of the cell
        const int ib = a + 1;                      // bottom row
        const bool border = (a == 0) && BY0;
        uint32_t acc = 0;
#pragma unroll
        for (int c = 1; c >= 0; --c) {     // cell column B first: it lands in the upper half of the word
            u64 top[2], bot[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                top[q] = c ? hB[it][q] : hA[it][q];
                bot[q] = c ? hB[ib][q] : hA[ib][q];
            }
#pragma unroll
            for (int ry = 3; ry >= 0; --ry) {
                const float h1f = border ? 0.0f : 0.125f + 0.25f * ry, h0f = 1.0f - h1f;
                const u64 h1 = pack2(h1f, h1f), h0 = pack2(h0f, h0f);
#pragma unroll
                for (int q = 1; q >= 0; --q) {
                    const u64 val = fma2(h0, top[q], mul2(h1, bot[q]));
                    const u64 d = fma2(val, NEG1, T0);   // T0 - val, one rounding
                    uint32_t dlo, dhi;
                    unpack2u(d, dlo, dhi);
                    acc = __funnelshift_l(dhi, acc, 1);
                    acc = __funnelshift_l(dlo, acc, 1);
                }
            }
        }
        word[a] = acc;
    }
    return ((u64)word[1] << 32) | word[0];
}
__device__ __forceinline__ u64 block_bits(const float (&v)[3][3], bool by0, bool bx0) {
    if (!by0 && !bx0) return block_bits_t<false, false>(v);
    if (by0 && !bx0) return block_bits_t<true, false>(v);
    if (!by0) return block_bits_t<false, true>(v);
    return block_bits_t<true, true>(v);
}

// =================================================================================================
// GT mask -> cell-block bits.  One CTA per (image, G_ROWS rows of blocks): the <= 8 * G_ROWS + 2 output rows it needs
// are one contiguous byte range; 32 pixels per job become one word of row bits (coalesced 32-byte reads, dot-product
// packing), then one thread per FOUR neighbouring blocks assembles their words with byte permutes.  Also clears the
// union words of the rows, the per-image accumulators and the work-queue counters.
// =================================================================================================
// 8 bytes -> 128 * (bit j = byte j != 0).  The carry trick leaves 0x80 in every non-zero byte; the 4-way byte dot
// product with the weights 1, 2, 4, ... then gathers the eight flags (no partial product overlaps another).
__device__ __forceinline__ uint32_t nz8_x128(uint32_t x0, uint32_t x1) {
    const uint32_t y0 = (((x0 & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x0) & 0x80808080u;
    const uint32_t y1 = (((x1 & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x1) & 0x80808080u;
    return __dp4a(y1, 0x80402010u, __dp4a(y0, 0x08040201u, 0u));
}
__device__ __forceinline__ uint32_t pack_u8x32(const uint4 &lo, const uint4 &hi) {
    const uint32_t g0 = nz8_x128(lo.x, lo.y), g1 = nz8_x128(lo.z, lo.w), g2 = nz8_x128(hi.x, hi.y), g3 = nz8_x128(hi.z, hi.w);
    return (g0 >> 7) | (g1 << 1) | (g2 << 9) | (g3 << 17);   // every g is a multiple of 128 below 2^15
}
__device__ __forceinline__ uint32_t pack_f32x32(const float4 *gp) {
    uint32_t bits = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float4 v = __ldg(gp + i);
        bits |= ((int)v.x != 0 ? 1u : 0u) << (4 * i) | ((int)v.y != 0 ? 1u : 0u) << (4 * i + 1) |
                ((int)v.z != 0 ? 1u : 0u) << (4 * i + 2) | ((int)v.w != 0 ? 1u : 0u) << (4 * i + 3);
    }
    return bits;
}
// Low nibbles of the four bytes of r -> 16 contiguous bits (byte k -> bits 4k .. 4k+3).
__device__ __forceinline__ uint32_t squeeze_nibbles(uint32_t r) {
    r = (r | (r >> 4)) & 0x00ff00ffu;
    return (r | (r >> 8)) & 0xffffu;
}

__global__ void __launch_bounds__(G_THREADS) gt_pack_kernel(const __grid_constant__ K3Params P) {
    // row bits of the CTA's output rows, flat: word q = pixels 32 (q % wpr) .. + 31 of row y_lo + q / wpr
    extern __shared__ uint32_t s_rows[];   // [(8 * G_ROWS + 2) * wpr]
    __shared__ int s_cnt[G_ROWS];
    const int by_lo = blockIdx.x * G_ROWS, b = blockIdx.y, tid = threadIdx.x;
    const int nby = min(G_ROWS, P.NBY - by_lo);
    const int S_h = P.S_h, S_w = P.S_w, wpr = S_w >> 5;
    const int y_lo = by_lo ? 8 * by_lo - 2 : 0, y_hi = min(8 * (by_lo + nby) - 2, S_h);   // output rows of these block rows
    const int nw = (y_hi - y_lo) * wpr;
    if (blockIdx.x == 0) {
        if (tid < 8) P.acc[b * 8 + tid] = 0;
        if (b == 0 && tid >= 32 && tid < 32 + 2 * C_NQ) P.work[((tid - 32) >> 1) * C_QSTRIDE + ((tid - 32) & 1)] = 0;   // detection / projector counters
    }
    if (tid < G_ROWS) s_cnt[tid] = 0;
    // ---- bytes -> row bits: the rows are contiguous in memory, job q = the q-th run of 32 pixels
    if (!P.gt_f32) {
        const uint4 *gp = reinterpret_cast<const uint4 *>(static_cast<const uint8_t *>(P.masks_gt) + ((size_t)b * S_h + y_lo) * S_w);
        constexpr int U = 3;   // jobs in flight per thread
        for (int q0 = tid; q0 < nw; q0 += U * G_THREADS) {
            uint4 v[U][2];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + u * G_THREADS;
                if (q < nw) { v[u][0] = __ldg(gp + 2 * q); v[u][1] = __ldg(gp + 2 * q + 1); }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + u * G_THREADS;
                if (q < nw) s_rows[q] = pack_u8x32(v[u][0], v[u][1]);
            }
        }
    } else {
        const float4 *gp = reinterpret_cast<const float4 *>(static_cast<const float *>(P.masks_gt) + ((size_t)b * S_h + y_lo) * S_w);
        for (int q = tid; q < nw; q += G_THREADS) s_rows[q] = pack_f32x32(gp + 8 * q);
    }
    __syncthreads();
    // ---- row bits -> block words.  Block (by, bx) is the 8 x 8 pixels at (8by - 2, 8bx - 2) of the zero-padded image:
    // shifted left by two pixels, a row of bits holds one BYTE per block, so a thread takes the 32-bit word of four
    // neighbouring blocks from each of the eight rows and transposes bytes into words with permutes.
    const int NBX = P.NBX, tpr = (NBX + 3) >> 2;   // threads per row of blocks
    for (int t = tid; t < nby * tpr; t += G_THREADS) {
        const int a_row = t / tpr, w = t - a_row * tpr, by = by_lo + a_row;
        uint32_t rw[8];
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
            const int y = 8 * by - 2 + rr;
            uint32_t prev = 0, cur = 0;
            if (y >= 0 && y < S_h) {
                const uint32_t *row = s_rows + (y - y_lo) * wpr;
                if (w > 0) prev = row[w - 1];
                if (w < wpr) cur = row[w];
            }
            rw[rr] = __funnelshift_r(prev, cur, 30);   // pixels 32w - 2 .. 32w + 29
        }
        const size_t o = ((size_t)b * P.NBY + by) * NBX + 4 * w;
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (4 * w + j >= NBX) break;
            // byte j of rows 0-3 / 4-7: pixels 0-3 of a row -> cell column A, 4-7 -> B; rows 0-3 -> cell row A, 4-7 -> B
            const uint32_t sel = (uint32_t)j | ((uint32_t)(4 + j) << 4);
            const uint32_t r03 = __byte_perm(__byte_perm(rw[0], rw[1], sel), __byte_perm(rw[2], rw[3], sel), 0x5410u);
            const uint32_t r47 = __byte_perm(__byte_perm(rw[4], rw[5], sel), __byte_perm(rw[6], rw[7], sel), 0x5410u);
            uint32_t lo = squeeze_nibbles(r03 & 0x0f0f0f0fu) | (squeeze_nibbles((r03 >> 4) & 0x0f0f0f0fu) << 16);
            uint32_t hi = squeeze_nibbles(r47 & 0x0f0f0f0fu) | (squeeze_nibbles((r47 >> 4) & 0x0f0f0f0fu) << 16);
            if (j == 0 && w == 0) {
                // block column 0: the border cell -1 owns the pixels x = 0, 1 as its columns 0, 1 (they sit at 2, 3 here)
                lo = (lo & 0xffff0000u) | ((lo >> 2) & 0x3333u);
                hi = (hi & 0xffff0000u) | ((hi >> 2) & 0x3333u);
            }
            if (by == 0) lo = (lo >> 8) & 0x00ff00ffu;   // block row 0: the border cell row owns y = 0, 1 as its rows 0, 1
            const u64 word = ((u64)hi << 32) | lo;
            P.gtc[o + j] = word;
            P.unc[o + j] = 0ull;
            cnt += __popc(lo) + __popc(hi);
        }
        if (cnt) atomicAdd(&s_cnt[a_row], cnt);
    }
    __syncthreads();
    if (tid < nby) P.gpart[b * P.NBY + by_lo + tid] = s_cnt[tid];
}

// =================================================================================================
// contract_kernel: one pass over the prototypes
// =================================================================================================
// BF16: the prototypes arrive as bfloat16 (the reference validates under bf16-mixed autocast and upcasts with
// .float()): a 16 KB tile with the 64-byte swizzle, widened exactly to fp32 on the way into the registers.
template <bool BF16>
__global__ void __launch_bounds__(A_THREADS, 4)
contract_kernel(const __grid_constant__ K3Params P, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(1024) unsigned char smem_dyn[];
    // the swizzled TMA destination must be 1024-byte aligned: align by hand (1024 spare bytes are allocated)
    unsigned char *smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    constexpr int TILE_FLOATS = NM * TA_H * TA_W / (BF16 ? 2 : 1);                     // tile size in 4-byte words
    float *s_tile = reinterpret_cast<float *>(smem);                                   // [NM][TA_H][TA_W], 16-byte chunks XOR row
    __shared__ __align__(8) uint64_t s_bar;
    // per-tile tables of the listed detections (coefficients, crop regions, pool offsets of the box origins), two sets:
    // the next tile's set is filled by cp.async while this tile is computed, so a tile costs ONE block barrier
    __shared__ __align__(16) float s_cf2[2][A_LCAP][NM];
    __shared__ __align__(8) short4 s_reg2[2][A_LCAP];
    __shared__ int s_off2[2][A_LCAP];
    __shared__ __align__(16) float s_w[NM];

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int tiles = P.ntx * P.nty, total = tiles * P.B;
    const int PH = P.PH, PW = P.PW, K = P.K;
    // this CTA's contiguous range of tiles (measured and not kept: tiles dealt round-robin to the CTAs, so that the grid
    // reads neighbouring tiles at the same time, 103.4 vs 100.5 us per pipelined step)
    const int t_begin = (int)(((long long)blockIdx.x * total) / gridDim.x);
    const int t_end = (int)(((long long)(blockIdx.x + 1) * total) / gridDim.x);
    if (t_begin >= t_end) return;

    // The tile buffer is dead as soon as every thread holds its pixels in registers: the next tile's TMA is issued
    // right then and lands under this tile's arithmetic (one buffer, four CTAs per SM).  Measured and not kept: two or
    // three buffers with three or two CTAs per SM (53.6 / 59.5 us: the kernel wants warps, not bytes in flight), and the
    // next 1 / 2 / 4 tiles prefetched into the L2 (101.5 / 102.6 / 106.6 vs 99.6 us per pipelined step).
    const bool keep_protos = __ldg(P.n_items + 1) != 0;
    // tile coordinates are stepped, not divided out, per tile (the divisions were a fifth of the kernel's instructions)
    struct TileAt { int b, ty, tx; };
    auto tile_at = [&](int tile) {
        TileAt a;
        a.b = tile / tiles;
        const int t = tile - a.b * tiles;
        a.ty = t / P.ntx; a.tx = t - a.ty * P.ntx;
        return a;
    };
    auto step = [&](TileAt &a) {   // to the next tile
        if (++a.tx == P.ntx) {
            a.tx = 0;
            if (++a.ty == P.nty) { a.ty = 0; ++a.b; }
        }
    };
    auto issue = [&](const TileAt &a) {   // thread 0
        mbar_expect_tx(&s_bar, (uint32_t)(TILE_FLOATS * sizeof(float)));
        tma_tile_g2s(s_tile, &tmap, a.tx * TA_W, a.ty * TA_H, a.b * NM, &s_bar, keep_protos);
    };
    TileAt at = tile_at(t_begin);   // current tile
    if (tid == 0) {
        mbar_init(&s_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        issue(at);
    }
    if (tid < NM) s_w[tid] = __ldg(P.proj_weight + tid);
    __syncthreads();

    // this thread's two pixels: rows {0,2,4,6} in lanes 0-15 and {1,3,5,7} in lanes 16-31 keep the 8-byte shared
    // loads of the swizzled tile free of bank conflicts
    const int i16 = lane & 15;
    const int row = 2 * (i16 >> 2) + (lane >> 4), colp = (wid << 3) + 2 * (i16 & 3);   // tile-local row / first column
    // fp32: 128-byte rows, chunk ^= row; bf16: 64-byte rows, chunk ^= (row >> 1) & 3 (offsets in 4-byte words)
    const int soff = BF16 ? row * (TA_W / 2) + ((((colp >> 3) ^ (row >> 1)) & 3) << 2) + ((colp & 7) >> 1)
                          : row * TA_W + (((colp >> 2) ^ row) << 2) + (colp & 3);

    // The tile's detections were binned by the plan.  List length and the list entries this thread copies are fetched
    // TWO tiles ahead; one tile ahead (right after the barrier that retires the previous tile's reads) every thread issues
    // its cp.async copies of the coefficients / regions / pool offsets into the other table set.
    struct Meta { int nlist, kq0, kq1, k0; };
    auto fetch_meta = [&](int tile) {
        Meta m;
        m.nlist = min(__ldg(P.tile_cnt + tile), K);
        const unsigned short *list = P.tile_list + (size_t)tile * K;
        const int nch0 = min(A_LCAP, m.nlist);
        m.kq0 = (tid < nch0 * (NM / 4)) ? __ldg(list + (tid >> 3)) : 0;
        m.kq1 = (tid + A_THREADS < nch0 * (NM / 4)) ? __ldg(list + ((tid + A_THREADS) >> 3)) : 0;
        m.k0 = (tid < nch0) ? __ldg(list + tid) : 0;
        return m;
    };
    auto stage_async = [&](const Meta &m, int b, int set) {   // round 0 of a tile's tables -> table set `set`
        const int nch0 = min(A_LCAP, m.nlist);
        if (tid < nch0 * (NM / 4))
            cp_async16(&s_cf2[set][tid >> 3][(tid & 7) * 4], P.det_coeff + ((size_t)b * K + m.kq0) * NM + (tid & 7) * 4);
        if (tid + A_THREADS < nch0 * (NM / 4))
            cp_async16(&s_cf2[set][(tid + A_THREADS) >> 3][(tid & 7) * 4], P.det_coeff + ((size_t)b * K + m.kq1) * NM + (tid & 7) * 4);
        if (tid < nch0) {
            cp_async8(&s_reg2[set][tid], P.det_region + (size_t)b * K + m.k0);
            cp_async4(&s_off2[set][tid], P.scr_off + (size_t)b * K + m.k0);
        }
    };
    Meta cur = fetch_meta(t_begin), nxt = cur;
    stage_async(cur, at.b, 0);
    if (t_begin + 1 < t_end) nxt = fetch_meta(t_begin + 1);

    for (int tile = t_begin, it = 0; tile < t_end; ++tile, ++it) {
        const int b = at.b;
        const int R0 = at.ty * TA_H, C0 = at.tx * TA_W;
        step(at);   // from here on `at` is the next tile
        const int r = R0 + row, c = C0 + colp;
        const int nlist = cur.nlist, set = it & 1;
        const unsigned short *list = P.tile_list + (size_t)tile * K;
        float (*s_cf)[NM] = s_cf2[set];
        short4 *s_reg = s_reg2[set];
        int *s_off = s_off2[set];

        // ---- the tile: shared memory -> registers, then the buffer is free for the next tile
        mbar_wait(&s_bar, (uint32_t)(it & 1));
        u64 p[NM];
        {
            const float *src = s_tile + soff;
            if (BF16) {
#pragma unroll
                for (int k = 0; k < NM; ++k) {
                    const uint32_t two = *reinterpret_cast<const uint32_t *>(src + k * (TA_H * TA_W / 2));
                    p[k] = ((u64)(two & 0xffff0000u) << 32) | (u64)(two << 16);   // bf16 -> fp32 is a 16-bit shift
                }
            } else {
#pragma unroll
                for (int k = 0; k < NM; ++k) p[k] = *reinterpret_cast<const u64 *>(src + k * (TA_H * TA_W));
            }
        }
        cp_async_wait_all();   // this thread's copies into the tile's table set (issued a tile ago)
        __syncthreads();       // the tile buffer is free, the table set is complete, the other set is no longer read
        if (tile + 1 < t_end) {
            if (tid == 0) issue(at);
            cur = nxt;
            stage_async(cur, at.b, set ^ 1);
            if (tile + 2 < t_end) nxt = fetch_meta(tile + 2);
        }

        // ---- M1 projection: bias + sum_k w_k p_k, sequential fma (== torch conv2d, pinned)
        {
            u64 acc = pack2(P.bias, P.bias);
#pragma unroll
            for (int k4 = 0; k4 < NM / 4; ++k4) {
                const float4 w4 = reinterpret_cast<const float4 *>(s_w)[k4];
                acc = fma2(pack2(w4.x, w4.x), p[4 * k4 + 0], acc);
                acc = fma2(pack2(w4.y, w4.y), p[4 * k4 + 1], acc);
                acc = fma2(pack2(w4.z, w4.z), p[4 * k4 + 2], acc);
                acc = fma2(pack2(w4.w, w4.w), p[4 * k4 + 3], acc);
            }
            // PW is even: both pixels of the pair are inside the image together
            if (r < PH && c < PW) *reinterpret_cast<u64 *>(P.lm + ((size_t)b * PH + r) * PW + c) = acc;
        }

        // ---- M2: rounds of A_LCAP listed detections
        const int wc0 = C0 + (wid << 3);   // the warp's 8 x 8 block: rows R0 .. R0+7, columns wc0 .. wc0+7
        for (int r0 = 0; r0 < nlist; r0 += A_LCAP) {
            const int nch = min(A_LCAP, nlist - r0);
            if (r0 > 0) {
                __syncthreads();   // the previous round's tables are still being read
                for (int q = tid; q < nch * (NM / 4); q += A_THREADS)
                    reinterpret_cast<float4 *>(&s_cf[q >> 3][0])[q & 7] =
                        __ldg(reinterpret_cast<const float4 *>(P.det_coeff + ((size_t)b * K + __ldg(list + r0 + (q >> 3))) * NM) + (q & 7));
                if (tid < nch) {
                    const int k = __ldg(list + r0 + tid);
                    const short4 rg = __ldg(P.det_region + (size_t)b * K + k);
                    s_reg[tid] = rg;
                    s_off[tid] = __ldg(P.scr_off + (size_t)b * K + k);
                }
                __syncthreads();
            }
            // the round's detections that touch this warp's block: one lane tests one detection
            short4 mine = make_short4(1, 0, 1, 0);
            if (lane < nch) mine = s_reg[lane];
            unsigned todo = __ballot_sync(0xffffffffu, lane < nch && mine.x <= R0 + TA_H - 1 && mine.y >= R0 && mine.z <= wc0 + 7 &&
                                                           mine.w >= wc0);
            auto store = [&](int e, u64 acc) {
                const short4 rg = s_reg[e];
                if (r >= rg.x && r <= rg.y) {
                    float a0, a1;
                    unpack2(acc, a0, a1);
                    float *dst = P.pool + (s_off[e] + (r - rg.x) * (rg.w - rg.z + 1) + (c - rg.z));
                    if (c >= rg.z && c <= rg.w) dst[0] = a0;
                    if (c + 1 >= rg.z && c + 1 <= rg.w) dst[1] = a1;
                }
            };
            // two detections at a time: two independent FFMA2 chains per thread
            while (todo & (todo - 1)) {
                const int e0 = __ffs(todo) - 1;
                todo &= todo - 1;
                const int e1 = __ffs(todo) - 1;
                todo &= todo - 1;
                u64 acc0 = pack2(0.0f, 0.0f), acc1 = acc0;
#pragma unroll
                for (int k4 = 0; k4 < NM / 4; ++k4) {
                    const float4 w0 = reinterpret_cast<const float4 *>(&s_cf[e0][0])[k4];
                    const float4 w1 = reinterpret_cast<const float4 *>(&s_cf[e1][0])[k4];
                    acc0 = fma2(pack2(w0.x, w0.x), p[4 * k4 + 0], acc0); acc1 = fma2(pack2(w1.x, w1.x), p[4 * k4 + 0], acc1);
                    acc0 = fma2(pack2(w0.y, w0.y), p[4 * k4 + 1], acc0); acc1 = fma2(pack2(w1.y, w1.y), p[4 * k4 + 1], acc1);
                    acc0 = fma2(pack2(w0.z, w0.z), p[4 * k4 + 2], acc0); acc1 = fma2(pack2(w1.z, w1.z), p[4 * k4 + 2], acc1);
                    acc0 = fma2(pack2(w0.w, w0.w), p[4 * k4 + 3], acc0); acc1 = fma2(pack2(w1.w, w1.w), p[4 * k4 + 3], acc1);
                }
                store(e0, acc0);
                store(e1, acc1);
            }
            if (todo) {
                const int e = __ffs(todo) - 1;
                u64 acc = pack2(0.0f, 0.0f);
#pragma unroll
                for (int k4 = 0; k4 < NM / 4; ++k4) {
                    const float4 w4 = reinterpret_cast<const float4 *>(&s_cf[e][0])[k4];
                    acc = fma2(pack2(w4.x, w4.x), p[4 * k4 + 0], acc);
                    acc = fma2(pack2(w4.y, w4.y), p[4 * k4 + 1], acc);
                    acc = fma2(pack2(w4.z, w4.z), p[4 * k4 + 2], acc);
                    acc = fma2(pack2(w4.w, w4.w), p[4 * k4 + 3], acc);
                }
                store(e, acc);
            }
        }
    }
}

// =================================================================================================
// cells_kernel: bilinear x4 + threshold + counters.  Persistent warps pull work items off one global counter:
// first the detections (one warp each, their sizes vary by 100x), then the projector mask in runs of 32 blocks.
// =================================================================================================
constexpr int C_WARPS = 4;   // warps per CTA of cells_kernel

__device__ __forceinline__ void m1_item(const K3Params &P, int b, int q, int lane) {
    const int PH = P.PH, PW = P.PW, S_h = P.S_h, S_w = P.S_w, NBX = P.NBX, NBY = P.NBY;
    int inter = 0, area = 0;
    double psum = 0.0;
    long long spt = 0, sp = 0;   // soft Dice: sum of p * t and of p over the valid pixels, units of 2^-40
    if (q < NBY * NBX) {
        int by = __float2int_rz(((float)q + 0.5f) * P.inv_NBX), bx = q - by * NBX;   // q / NBX without the integer division
        if (bx < 0) { --by; bx += NBX; } else if (bx >= NBX) { ++by; bx -= NBX; }
        const BlockGeo g = block_geo(by, bx, PH, PW);
        const float *lm = P.lm + (size_t)b * PH * PW;
        float v[3][3];
        const int rr[3] = {g.r0 * PW, g.r1 * PW, g.r2 * PW}, cc[3] = {g.c0, g.c1, g.c2};
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) v[i][j] = __ldg(lm + rr[i] + cc[j]);
        const u64 gtw = __ldg(P.gtc + ((size_t)b * NBY + by) * NBX + bx);
        if (!(P.seg_logits || P.seg_mask || P.seg_prob_sum || P.seg_soft2)) {
            const u64 bits = block_bits(v, by == 0, bx == 0) & block_valid(P, by, bx);
            area = __popcll(bits); inter = __popcll(bits & gtw);
        } else {
            // dense outputs / v3 score / soft Dice: scalar path that keeps the logits
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const int ci = 2 * by - 1 + a, cj = 2 * bx - 1 + c;
                    if (ci > PH - 1 || cj > PW - 1) continue;
                    const int it = (a == 0 || by == 0) ? 0 : 1, ib = (a == 0) ? 1 : 2;
                    const int jl = (c == 0 || bx == 0) ? 0 : 1, jr = (c == 0) ? 1 : 2;
                    float lg[16];
                    unsigned bits = cell_bits_log(v[it][jl], v[it][jr], v[ib][jl], v[ib][jr], ci < 0, cj < 0, lg);
                    const unsigned valid = cell_valid(ci, cj, PH, PW, S_h, S_w);
                    const unsigned gt = (unsigned)((gtw >> (16 * (2 * a + c))) & 0xffffull);
                    bits &= valid;
                    area += __popc(bits);
                    inter += __popc(bits & gt);
                    if (P.seg_soft2) {
#pragma unroll
                        for (int k = 0; k < 16; ++k)
                            if ((valid >> k) & 1u) {
                                const long long pf = soft_prob_fx40(lg[k]);
                                sp += pf;
                                if ((gt >> k) & 1u) spt += pf;
                            }
                    }
                    if (P.seg_prob_sum && bits) {
                        float ps = 0.0f;   // v3 seg-mAP score numerator: sigmoid over the foreground pixels of the cell
#pragma unroll
                        for (int k = 0; k < 16; ++k)
                            if ((bits >> k) & 1u) ps += 1.0f / (1.0f + __expf(-lg[k]));
                        psum += (double)ps;
                    }
                    if (P.seg_logits || P.seg_mask) {
                        const int ybase = (ci < 0) ? 0 : 4 * ci + 2, xbase = (cj < 0) ? 0 : 4 * cj + 2;
                        const int nry = (ci < 0) ? 2 : min(4, S_h - ybase), nrx = (cj < 0) ? 2 : min(4, S_w - xbase);
#pragma unroll
                        for (int ry = 0; ry < 4; ++ry) {
                            if (ry >= nry) break;
                            const size_t o = ((size_t)b * S_h + ybase + ry) * S_w + xbase;
#pragma unroll
                            for (int rx = 0; rx < 4; ++rx) {
                                if (rx >= nrx) break;
                                if (P.seg_logits) P.seg_logits[o + rx] = lg[ry * 4 + rx];
                                if (P.seg_mask) P.seg_mask[o + rx] = (bits >> (ry * 4 + rx)) & 1u;
                            }
                        }
                    }
                }
        }
    }
    inter = __reduce_add_sync(0xffffffffu, inter);
    area = __reduce_add_sync(0xffffffffu, area);
    if (lane == 0) {
        if (inter) atomicAdd(&P.acc[b * 8 + 0], inter);
        if (area) atomicAdd(&P.acc[b * 8 + 1], area);
    }
    if (P.seg_prob_sum) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) psum += __shfl_down_sync(0xffffffffu, psum, d);
        if (lane == 0 && psum != 0.0) atomicAdd(&P.seg_prob_sum[b], psum);
    }
    if (P.seg_soft2) {   // integer sums: exact, so the order of the lanes and of the items does not matter
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            spt += __shfl_down_sync(0xffffffffu, spt, d);
            sp += __shfl_down_sync(0xffffffffu, sp, d);
        }
        if (lane == 0) {
            unsigned long long *s2 = reinterpret_cast<unsigned long long *>(P.seg_soft2 + 2 * b);
            if (spt) atomicAdd(s2, (unsigned long long)spt);
            if (sp) atomicAdd(s2 + 1, (unsigned long long)sp);
        }
    }
}

// =================================================================================================
// seg_curve_kernel (btpost_seg_curve): binned precision-recall / ROC state of the projector probabilities.  Reads the
// projector logits at prototype resolution and the GT block words that btpost_masks left in the workspace, redoes
// m1_item's bilinear x4 per 2x2 cell block (block_geo / cell_bits_log / cell_valid: the logits of cells_kernel, bit for
// bit), and counts every valid pixel in hist[t][j], t = its GT bit, j = the number of thresholds <= p = soft_prob(x).
// =================================================================================================
// A persistent grid of 3 CTAs per SM (up to 85 registers; at 4, ptxas spills), few enough CTAs that the flush (at most
// 2 (T + 1) atomics per CTA) stays small; each thread takes one block (<= 64 pixels) at a time, grid-strided
constexpr int CV_THREADS = 256, CV_CTAS_PER_SM = 3;
constexpr int CV_LUT = 2048;   // cells of the threshold table

struct CurveParams {
    int B, S_h, S_w, PH, PW, NBY, NBX;
    int T;                  // thresholds
    int span;               // power of two > T (building the threshold table)
    const float *lm;        // [B, PH, PW] projector logits (workspace)
    const u64 *gtc;         // [B, NBY, NBX] GT bits per 2x2 block of cells (workspace)
    unsigned long long *hist;   // [2, T + 1], accumulated
    float thr[BT_MAX_CURVE_THRS];   // non-decreasing, in [0, 1] (checked by the entry point)
};

// Finding j: a table over CV_LUT equal cells of [0, 1] gives, for the cell of p, the thresholds below the cell (all <= p)
// and those in it; a search over the few in the cell finishes (one or two compares for linspace thresholds, at most
// log2(T) whatever the list).
// Counting: neighbouring pixels of a lane's block mostly fall in one bin, so a lane counts its run of equal bins in a
// register and adds the run to the CTA's u32 bins in shared memory with one atomic when the bin changes (measured on a
// B200 at 64 x 640^2, T = 101: 128 us, against 202 us with a warp match per pixel and one atomic per distinct bin).  The
// CTA's bins go to `hist` once, with one 64-bit atomic per non-zero bin.  Integer sums: the words do not depend on the
// launch shape.
__global__ void __launch_bounds__(CV_THREADS, CV_CTAS_PER_SM) seg_curve_kernel(const __grid_constant__ CurveParams P) {
    __shared__ float s_thr[BT_MAX_CURVE_THRS];
    __shared__ unsigned short s_lut[CV_LUT + 2];   // s_lut[c] = thresholds < c / CV_LUT (c <= CV_LUT); s_lut[CV_LUT + 1] = T
    __shared__ uint32_t s_hist[2 * (BT_MAX_CURVE_THRS + 1)];
    const int T = P.T, nbins = 2 * (T + 1);
    for (int i = threadIdx.x; i < T; i += CV_THREADS) s_thr[i] = P.thr[i];
    for (int i = threadIdx.x; i < nbins; i += CV_THREADS) s_hist[i] = 0u;
    __syncthreads();
    for (int c = threadIdx.x; c < CV_LUT + 2; c += CV_THREADS) {
        const float lo = (float)c * (1.0f / CV_LUT);   // exact
        int n = 0;
        for (int step = P.span >> 1; step > 0; step >>= 1)
            if (n + step <= T && s_thr[n + step - 1] < lo) n += step;
        s_lut[c] = (unsigned short)(c == CV_LUT + 1 ? T : n);
    }
    __syncthreads();
    const int PH = P.PH, PW = P.PW, NBX = P.NBX;
    const long long per_image = (long long)P.NBY * NBX, total = P.B * per_image;
    const long long stride = (long long)gridDim.x * CV_THREADS;
    uint32_t run_key = 0u, run_n = 0u;   // this lane's current run of pixels in one bin
    for (long long q = (long long)blockIdx.x * CV_THREADS + threadIdx.x; q < total; q += stride) {
        int by = 0, bx = 0;
        float v[3][3];
        u64 gtw;
        {
            const int b = (int)(q / per_image), r = (int)(q - b * per_image);
            by = r / NBX; bx = r - by * NBX;
            const BlockGeo g = block_geo(by, bx, PH, PW);
            const float *lm = P.lm + (size_t)b * PH * PW;
            const int rr[3] = {g.r0 * PW, g.r1 * PW, g.r2 * PW}, cc[3] = {g.c0, g.c1, g.c2};
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) v[i][j] = __ldg(lm + rr[i] + cc[j]);
            gtw = __ldg(P.gtc + q);
        }
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int ci = 2 * by - 1 + a, cj = 2 * bx - 1 + c;
                // m1_item's corners v[it][jl] .. v[ib][jr] as selects (a runtime index would put v in local memory)
                const bool up = a == 1 && by != 0, left = c == 1 && bx != 0;
                const float v00 = up ? (left ? v[1][1] : v[1][0]) : (left ? v[0][1] : v[0][0]);
                const float v01 = up ? v[1][c + 1] : v[0][c + 1];
                const float v10 = left ? v[a + 1][1] : v[a + 1][0];
                float lg[16];
                cell_bits_log(v00, v01, v10, v[a + 1][c + 1], ci < 0, cj < 0, lg);
                const unsigned valid = cell_valid(ci, cj, PH, PW, P.S_h, P.S_w);
                const unsigned gt = (unsigned)(gtw >> (16 * (2 * a + c))) & 0xffffu;
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const float p = soft_prob(lg[k]);
                    // thresholds <= p: those below p's cell, then a search among the cell's own (a NaN p: cell 0, j = 0)
                    const int cell = p == p ? (int)__fmul_rn(p, (float)CV_LUT) : 0;   // p in [0, 1]
                    int j = s_lut[cell], n = s_lut[cell + 1] - j;
                    while (n > 0) {
                        const int h = n >> 1;
                        if (s_thr[j + h] <= p) { j += h + 1; n -= h + 1; } else { n = h; }
                    }
                    const uint32_t key = ((gt >> k) & 1u) * (uint32_t)(T + 1) + (uint32_t)j;
                    if ((valid >> k) & 1u) {
                        if (key != run_key) {
                            if (run_n) atomicAdd(&s_hist[run_key], run_n);
                            run_key = key; run_n = 0u;
                        }
                        ++run_n;
                    }
                }
            }
    }
    if (run_n) atomicAdd(&s_hist[run_key], run_n);
    __syncthreads();
    for (int i = threadIdx.x; i < nbins; i += CV_THREADS)
        if (const uint32_t n = s_hist[i]) atomicAdd(P.hist + i, (unsigned long long)n);
}

// Optional output: the block's 8 x 8 pixels into the detection's bit-packed plane (zeroed beforehand).  A block row is
// 8 pixels starting at x = 8bx - 2 (6 pixels at x = 0 for bx = 0), so it shares its 32-bit word with the neighbouring
// blocks: fire-and-forget atomic ORs (RED) into the L2.  Pixels outside the image are already masked out of `bits`.
__device__ __forceinline__ void scatter_block_bits(const K3Params &P, int bk, int by, int bx, u64 bits) {
    const int wpr = P.S_w >> 5;
    uint32_t *plane = P.inst_bits + (size_t)bk * P.S_h * wpr;
    const int xb = bx ? 8 * bx - 2 : 0, sh = xb & 31;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const int ci = 2 * by - 1 + a, ybase = ci < 0 ? 0 : 4 * ci + 2;
        const unsigned cellA = (unsigned)(bits >> (32 * a)) & 0xffffu, cellB = (unsigned)(bits >> (32 * a + 16)) & 0xffffu;
        if (!(cellA | cellB)) continue;
#pragma unroll
        for (int ry = 0; ry < 4; ++ry) {
            const unsigned nA = (cellA >> (4 * ry)) & 0xfu, nB = (cellB >> (4 * ry)) & 0xfu;
            const unsigned row8 = bx ? (nA | (nB << 4)) : (nA | (nB << 2));   // bx = 0: the border cell holds 2 pixels
            if (!row8) continue;
            uint32_t *w = plane + (size_t)(ybase + ry) * wpr + (xb >> 5);
            atomicOr(w, row8 << sh);
            if (sh > 24 && (row8 >> (32 - sh))) atomicOr(w + 1, row8 >> (32 - sh));   // never past the row: those pixels are masked out
        }
    }
}

// One item of a detection = blocks [chunk * C_CHUNK, (chunk + 1) * C_CHUNK) of its crop box (the plan lists them).
// An item is worked on by a GROUP of GS lanes, GS blocks per pass: the crop boxes of the benchmark's detections hold
// 28 blocks on average (median 24), so whole-warp passes ran at 65 % lane utilisation; groups of 8 lanes reach 94 %.
// The groups of a warp hold different detections; everything per item lives in the lanes' own registers.
struct DetWork {
    int bk, b, i, i_end, off, nbx;
    short4 rg;       // crop region at prototype resolution (r_lo, r_hi, c_lo, c_hi)
    float inv;       // 1 / nbx
};
__device__ __forceinline__ void det_begin(const K3Params &P, int bk, int chunk, DetWork &w) {
    const int K = P.K;
    int b = __float2int_rz(((float)bk + 0.5f) * P.inv_K), k = bk - b * K;
    if (k < 0) --b; else if (k >= K) ++b;
    const short4 rg = __ldg(P.det_region + bk);
    const int nbx = ((rg.w + 1) >> 1) - (rg.z >> 1) + 1, nby = ((rg.y + 1) >> 1) - (rg.x >> 1) + 1;
    w.bk = bk; w.b = b; w.rg = rg; w.nbx = nbx;
    w.i = chunk * C_CHUNK;
    w.i_end = min(nbx * nby, (chunk + 1) * C_CHUNK);
    w.off = __ldg(P.scr_off + bk);
    w.inv = __fdividef(1.0f, (float)nbx);   // approximate is enough: det_pass repairs a quotient that is off by one
}
// one pass: block w.i + gl of the item (gl = lane within the group)
template <int GS>
__device__ __forceinline__ void det_pass(const K3Params &P, const DetWork &w, int gl, unsigned gmask, int gbase, int &area, int &inter,
                                         int &uarea, int &uinter) {
    const int PH = P.PH, PW = P.PW, NBX = P.NBX, NBY = P.NBY;
    const int r_lo = w.rg.x, r_hi = w.rg.y, c_lo = w.rg.z, c_hi = w.rg.w, bw = c_hi - c_lo + 1;
    const int by0 = r_lo >> 1, bx0 = c_lo >> 1, nbx = w.nbx, b = w.b;
    const int i = w.i + gl;
    const bool act = i < w.i_end;
    int yy = __float2int_rz(((float)i + 0.5f) * w.inv);
    int xx = i - yy * nbx;
    if (xx < 0) { --yy; xx += nbx; } else if (xx >= nbx) { ++yy; xx -= nbx; }
    const int by = act ? by0 + yy : by0, bx = act ? bx0 + xx : bx0;
    const BlockGeo g = block_geo(by, bx, PH, PW);
    const int rr[3] = {g.r0, g.r1, g.r2}, cc[3] = {g.c0, g.c1, g.c2};
    bool rin[3], cin[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        rin[a] = act && rr[a] >= r_lo && rr[a] <= r_hi;
        cin[a] = cc[a] >= c_lo && cc[a] <= c_hi;
    }
    float v[3][3];
    if (w.off >= 0) {
        // the crop box's logits; corners outside the box are zero (clamped address, value discarded)
        const float *scr = P.pool + w.off;
        int ro[3], co[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            ro[a] = (min(max(rr[a], r_lo), r_hi) - r_lo) * bw;
            co[a] = min(max(cc[a], c_lo), c_hi) - c_lo;
        }
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float x = __ldg(scr + ro[a] + co[c]);
                v[a][c] = (rin[a] && cin[c]) ? x : 0.0f;
            }
    } else {
        // no room in the logit pool (huge crop boxes / crop off): contract the 9 corners here, same sequential order;
        // the group's lanes hold the 32 coefficients between them and broadcast one per channel with a shuffle
        constexpr int NPL = NM / GS;
        const float *cf = P.det_coeff + (size_t)w.bk * NM;
        float mycf[NPL];
#pragma unroll
        for (int q = 0; q < NPL; ++q) mycf[q] = __ldg(cf + q * GS + gl);
        const size_t pr0 = (size_t)b * NM * PH * PW;
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int c = 0; c < 3; ++c) v[a][c] = 0.0f;
        if (!P.proto_bf16) {
            const float *pr = static_cast<const float *>(P.protos) + pr0;
#pragma unroll
            for (int q = 0; q < NPL; ++q)
                for (int cl = 0; cl < GS; ++cl) {
                    const float wt = __shfl_sync(gmask, mycf[q], gbase + cl);
                    const float *pc = pr + (size_t)(q * GS + cl) * PH * PW;
#pragma unroll
                    for (int a = 0; a < 3; ++a)
#pragma unroll
                        for (int c = 0; c < 3; ++c)
                            if (rin[a] && cin[c]) v[a][c] = __fmaf_rn(wt, __ldg(pc + rr[a] * PW + cc[c]), v[a][c]);
                }
        } else {
            const unsigned short *pr = static_cast<const unsigned short *>(P.protos) + pr0;
#pragma unroll
            for (int q = 0; q < NPL; ++q)
                for (int cl = 0; cl < GS; ++cl) {
                    const float wt = __shfl_sync(gmask, mycf[q], gbase + cl);
                    const unsigned short *pc = pr + (size_t)(q * GS + cl) * PH * PW;
#pragma unroll
                    for (int a = 0; a < 3; ++a)
#pragma unroll
                        for (int c = 0; c < 3; ++c)
                            if (rin[a] && cin[c])
                                v[a][c] = __fmaf_rn(wt, __uint_as_float((uint32_t)__ldg(pc + rr[a] * PW + cc[c]) << 16), v[a][c]);
                }
        }
    }
    const size_t o = ((size_t)b * NBY + by) * NBX + bx;
    const u64 gtw = __ldg(P.gtc + o);   // with the corner loads, not behind the arithmetic
    if (!act) return;
    const u64 bits = block_bits(v, by == 0, bx == 0) & block_valid(P, by, bx);
    if (bits && P.inst_bits) scatter_block_bits(P, w.bk, by, bx, bits);
    if (bits) {
        // the OR is serialised per word in the L2: the bits that were not set before are counted exactly once
        // over all detections, so the union's counters need no pass over the union afterwards
        const u64 fresh = bits & ~atomicOr(P.unc + o, bits);
        area += __popcll(bits);
        inter += __popcll(bits & gtw);
        uarea += __popcll(fresh);
        uinter += __popcll(fresh & gtw);
    }
}
// item done: the group's sums (one REDUX each) -> the detection's / the image's counters
__device__ __forceinline__ void det_end(const K3Params &P, const DetWork &w, unsigned gmask, int gl, int area, int inter, int uarea,
                                        int uinter) {
    inter = __reduce_add_sync(gmask, inter);
    area = __reduce_add_sync(gmask, area);
    uinter = __reduce_add_sync(gmask, uinter);
    uarea = __reduce_add_sync(gmask, uarea);
    if (gl == 0) {
        // zeroed by the NMS kernel; a detection of several chunks adds up
        if (P.inst_area && area) atomicAdd(&P.inst_area[w.bk], area);
        if (P.inst_inter && inter) atomicAdd(&P.inst_inter[w.bk], inter);
        if (uinter) atomicAdd(&P.acc[w.b * 8 + 3], uinter);
        if (uarea) atomicAdd(&P.acc[w.b * 8 + 4], uarea);
    }
}

// v3 segmentation-mAP record of image b (running_main_v3.py:478-498): the projector mask, scored by its mean foreground
// probability, against the GT mask, class 0 -- what btpost/segmap.py builds from the same outputs, for COCOeval with one
// detection and one GT per image.  seg_prob_sum is exact in double: each addend is an fp32 per-cell sum of
// probabilities >= 0.5, hence a multiple of 2^-24, and the total stays below 2^20 even at 1024^2, so every partial sum
// fits in 44 bits.  The score therefore depends neither on the order of m1_item's atomics nor on the sharding.
__device__ __forceinline__ void seg_map_record(const K3Params &P, int b, long long inter, long long pp, long long gsum) {
    long long *hdr = P.seg_sweep;
    const int T = P.T;
    const float score = __fdiv_rn(__double2float_rn(__ldcg(P.seg_prob_sum + b)), __fadd_rn((float)pp, 1e-6f));
    const long long uni = pp + gsum - inter;
    const double iou = uni > 0 ? (double)inter / (double)uni : 0.0;
    const unsigned long long tmask = (T >= 16) ? 0xffffull : ((1ull << T) - 1ull);
    unsigned long long hit = 0ull;
    for (int t = 0; t < T; ++t) hit |= (iou >= fmin(P.thrs[t], 1 - 1e-10) ? 1ull : 0ull) << t;
    const double area_lo[BT_NUM_AREA] = COCO_AREA_LO;
    const double area_hi[BT_NUM_AREA] = COCO_AREA_HI;
    unsigned long long matched = 0ull, ignored = 0ull;
#pragma unroll
    for (int a = 0; a < BT_NUM_AREA; ++a) {
        const bool gt_ig = (double)gsum < area_lo[a] || (double)gsum > area_hi[a];
        const bool dt_out = (double)pp < area_lo[a] || (double)pp > area_hi[a];
        matched |= hit << (a * T);
        ignored |= ((gt_ig ? hit : 0ull) | (dt_out ? (~hit & tmask) : 0ull)) << (a * T);   // a hit takes the GT's flag
        if (!gt_ig) atomicAdd(reinterpret_cast<unsigned long long *>(hdr + BT_SWEEP_NPIG + a * BT_MAX_CLASSES), 1ull);
    }
    atomicAdd(reinterpret_cast<unsigned long long *>(hdr + BT_SWEEP_N_IMAGES), 1ull);
    const long long pos = (long long)atomicAdd(reinterpret_cast<unsigned long long *>(hdr + BT_SWEEP_N_RECORDS), 1ull);
    if (pos >= __ldcg(hdr + BT_SWEEP_CAPACITY)) return;   // ring full: reported through the header (N_RECORDS > CAPACITY)
    BtSweepRecord r;
    r.matched = matched;
    r.ignored = ignored;
    r.score_key = desc_key(score);
    r.image = (uint32_t)(P.image_offset + (P.image_base ? __ldg(P.image_base) : 0) + b);
    r.rank = 0; r.class_rank = 0; r.label = 0;
    r.pad[0] = r.pad[1] = r.pad[2] = 0;
    uint4 *dst = reinterpret_cast<uint4 *>(reinterpret_cast<BtSweepRecord *>(hdr + BT_SWEEP_HEADER_I64) + pos);
    const uint4 *src = reinterpret_cast<const uint4 *>(&r);
    dst[0] = src[0];
    dst[1] = src[1];
}

// v3 soft Dice of image b (SURVEY.md A.4; DiceScore on the projector probabilities, running_main_v3.py:466-474):
// 2 A / (P + G) with A = sum p * t and P = sum p from m1_item's 2^-40 sums and G = |G|, in double, rounded to fp32;
// NaN (and left out of the accumulator's count) when P + G == 0, as the reference's mean skips NaN.
__device__ __forceinline__ void soft_dice_image(const K3Params &P, int b, long long gsum) {
    const long long a = __ldcg(P.seg_soft2 + 2 * b), p = __ldcg(P.seg_soft2 + 2 * b + 1);
    const bool defined = p != 0 || gsum != 0;
    const float d = defined ? __double2float_rn(2.0 * (double)a / ((double)p + (double)gsum * 1099511627776.0))
                            : __int_as_float(0x7fc00000);
    if (P.seg_soft_dice) P.seg_soft_dice[b] = d;
    if (P.seg_soft_acc && defined) {
        unsigned long long *acc = reinterpret_cast<unsigned long long *>(P.seg_soft_acc);
        atomicAdd(acc, (unsigned long long)__double2ll_rn((double)d * 1099511627776.0));
        atomicAdd(acc + 1, 1ull);
    }
}

// per-image epilogue: |G|, Dice / IoU (test_model.py:15-23)
__device__ __forceinline__ void finalize_image(const K3Params &P, int b, int lane) {
    int gg = 0;
    for (int q = lane; q < P.NBY; q += 32) gg += __ldcg(P.gpart + b * P.NBY + q);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) gg += __shfl_xor_sync(0xffffffffu, gg, d);
    if (lane < 2) {
        const long long inter = __ldcg(P.acc + b * 8 + 3 * lane), pp = __ldcg(P.acc + b * 8 + 3 * lane + 1), gsum = gg;
        const long long total = (long long)P.S_h * P.S_w;
        long long *img3 = lane ? P.uni_img3 : P.seg_img3;
        long long *cnt4 = lane ? P.uni_cnt4 : P.seg_cnt4;
        float *dice = lane ? P.uni_dice : P.seg_dice, *iou = lane ? P.uni_iou : P.seg_iou;
        if (img3) { img3[b * 3 + 0] = inter; img3[b * 3 + 1] = pp; img3[b * 3 + 2] = gsum; }
        if (cnt4) {
            atomicAdd((unsigned long long *)&cnt4[0], (unsigned long long)inter);
            atomicAdd((unsigned long long *)&cnt4[1], (unsigned long long)(pp - inter));
            atomicAdd((unsigned long long *)&cnt4[2], (unsigned long long)(gsum - inter));
            atomicAdd((unsigned long long *)&cnt4[3], (unsigned long long)(total - pp - gsum + inter));
        }
        const float fi = (float)inter, fu = (float)(pp + gsum - inter);
        const float v_iou = __fdiv_rn(__fadd_rn(fi, 1e-7f), __fadd_rn(fu, 1e-7f));
        const float v_dice = __fdiv_rn(__fadd_rn(__fmul_rn(2.0f, fi), 1e-7f), __fadd_rn(__fadd_rn((float)pp, (float)gsum), 1e-7f));
        if (iou) iou[b] = v_iou;
        if (dice) dice[b] = v_dice;
        if (P.sweep) {   // order-independent sums: 2^-40 fixed point (the values are in [0, 1])
            unsigned long long *fs = reinterpret_cast<unsigned long long *>(P.sweep + BT_SWEEP_FSUM + 2 * lane);
            atomicAdd(fs, (unsigned long long)__double2ll_rn((double)v_dice * 1099511627776.0));
            atomicAdd(fs + 1, (unsigned long long)__double2ll_rn((double)v_iou * 1099511627776.0));
        }
        if (lane == 0 && P.seg_sweep) seg_map_record(P, b, inter, pp, gsum);
        if (lane == 0 && P.seg_soft2) soft_dice_image(P, b, gsum);
    }
}

__device__ __forceinline__ int atom_inc(int *p) {
    int v;
    asm volatile("atom.global.add.u32 %0, [%1], 1;" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Work queues: item i lives in queue i % nq; one counter per queue and kind of item (detections / projector runs), a
// queue's counters in one 128-byte line of their own (atomics on one address serialise in the L2: a single counter took
// 2 ns per item, the whole kernel's time).  A warp serves its home queue until it is drained and then leaves: every queue
// holds the same mix of items and has the same number of warps, so they drain together (stealing from the other queues
// cost a scan of 31 counters per warp at the end).  Detection items are taken by lane GROUPS (see DetWork), the projector
// mask's runs of 32 blocks by whole warps once the queue's detections are out.
// The detection items of queue q, taken by groups of GS lanes.
template <int GS>
__device__ __forceinline__ void det_phase(const K3Params &P, int q, int ndet, int lane) {
    const int gl = lane & (GS - 1), gbase = lane & ~(GS - 1);
    const unsigned gmask = GS == 32 ? 0xffffffffu : (((1u << GS) - 1u) << gbase);
    int *ctr = P.work + q * C_QSTRIDE;
    int j = 0;
    if (gl == 0) j = atom_inc(ctr);
    bool have = false, done = false;
    DetWork w{};
    int area = 0, inter = 0, uarea = 0, uinter = 0;   // uarea / uinter: pixels this detection ADDS to the image's union
    for (;;) {
        if (!have && !done) {
            const int item = q + P.nq * __shfl_sync(gmask, j, gbase);
            if (item < ndet) {
                if (gl == 0) j = atom_inc(ctr);   // next item of the queue: in flight while this one is processed
                const int2 it = __ldg(P.items + item);
                det_begin(P, it.x, it.y, w);
                have = true;
            } else {
                done = true;
            }
        }
        if (__all_sync(0xffffffffu, done)) break;
        if (have) {
            det_pass<GS>(P, w, gl, gmask, gbase, area, inter, uarea, uinter);
            w.i += GS;
            if (w.i >= w.i_end) {
                det_end(P, w, gmask, gl, area, inter, uarea, uinter);
                area = inter = uarea = uinter = 0;
                have = false;
            }
        }
    }
}

__global__ void __launch_bounds__(C_WARPS * 32, 8) cells_kernel(const __grid_constant__ K3Params P) {
    const int lane = threadIdx.x & 31;
    const int ndet = min(__ldg(P.n_items), P.item_cap);
    const int q = (blockIdx.x * C_WARPS + (threadIdx.x >> 5)) & (P.nq - 1);
    // Detection items are taken by groups of 16 lanes (measured and not kept, pipelined step: groups of 32 / 8 / 4 lanes
    // = 99.4 / 101.1 / 108.4 us against 97.4 us for 16).  Some detection found no room in the logit pool (huge crop
    // boxes / crop off): its items contract their corners from the prototypes, 32 channels x 9 loads per block; that path
    // runs best with whole-warp items (measured: L1 layout with random DFL boxes, mask stage 519 us with whole warps,
    // 685 us with groups of 16).
    if (__ldg(P.n_items + 1) != 0) det_phase<32>(P, q, ndet, lane);
    else det_phase<16>(P, q, ndet, lane);
    {
        const int total = P.B * P.m1_items;
        int *ctr = P.work + q * C_QSTRIDE + 1;
        int j = 0;
        if (lane == 0) j = atom_inc(ctr);
        for (;;) {
            const int m = __shfl_sync(0xffffffffu, q + P.nq * j, 0);
            if (m >= total) break;
            if (lane == 0) j = atom_inc(ctr);
            int b = __float2int_rz(((float)m + 0.5f) * P.inv_m1);
            int c = m - b * P.m1_items;
            if (c < 0) { --b; c += P.m1_items; } else if (c >= P.m1_items) { ++b; c -= P.m1_items; }
            m1_item(P, b, c * 32 + lane, lane);
        }
    }
}

// per-image epilogue, one warp per image: |G|, Dice / IoU (test_model.py:15-23)
__global__ void __launch_bounds__(C_THREADS) finalize_kernel(const __grid_constant__ K3Params P) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * (C_THREADS / 32) + (threadIdx.x >> 5);
    if (b < P.B) finalize_image(P, b, lane);
}

// optional dense output: union words -> bytes
__global__ void __launch_bounds__(C_THREADS) union_dense_kernel(const __grid_constant__ K3Params P) {
    const int b = blockIdx.x, tid = threadIdx.x;
    const u64 *un = P.unc + (size_t)b * P.NBY * P.NBX;
    const int S_h = P.S_h, S_w = P.S_w;
    // thread = (output row, block), 8 pixels of that row (6 in block column 0)
    for (int q = tid; q < S_h * P.NBX; q += C_THREADS) {
        const int y = q / P.NBX, bx = q - y * P.NBX;
        const int ci = (y < 2) ? -1 : (y - 2) >> 2, ry = (y < 2) ? y : (y - 2) & 3;
        const int by = (ci + 1) >> 1, a = (ci + 1) & 1;
        const u64 w = __ldg(un + (size_t)by * P.NBX + bx);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const int cj = 2 * bx - 1 + c;
            if (cj > P.PW - 1) continue;
            const int xbase = (cj < 0) ? 0 : 4 * cj + 2, nrx = (cj < 0) ? 2 : min(4, S_w - xbase);
            const unsigned nib = (unsigned)(w >> (16 * (2 * a + c) + 4 * ry)) & 0xfu;
            uint8_t *o = P.uni_mask + ((size_t)b * S_h + y) * S_w + xbase;   // 2-byte aligned
            *reinterpret_cast<uchar2 *>(o) = make_uchar2(nib & 1u, (nib >> 1) & 1u);
            if (nrx == 4) *reinterpret_cast<uchar2 *>(o + 2) = make_uchar2((nib >> 2) & 1u, (nib >> 3) & 1u);
        }
    }
}

// optional dense output: bit-packed instance masks -> bytes {0,1}; one 32-pixel word per thread, 32 contiguous bytes out
__global__ void __launch_bounds__(C_THREADS) inst_dense_kernel(const uint32_t *__restrict__ bits, uint8_t *__restrict__ out,
                                                               size_t nwords) {
    for (size_t i = (size_t)blockIdx.x * C_THREADS + threadIdx.x; i < nwords; i += (size_t)gridDim.x * C_THREADS) {
        const uint32_t w = __ldg(bits + i);
        uint4 o[2];
        uint32_t *ow = reinterpret_cast<uint32_t *>(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t n = (w >> (4 * j)) & 0xfu;   // 4 pixels -> 4 bytes
            ow[j] = (n & 1u) | ((n & 2u) << 7) | ((n & 4u) << 14) | ((n & 8u) << 21);
        }
        uint4 *dst = reinterpret_cast<uint4 *>(out + i * 32);
        __stcs(dst, o[0]);
        __stcs(dst + 1, o[1]);
    }
}

// 3-D tensor map of the prototypes: dims (fastest first) {PW, PH, B*NM}, box {TA_W, TA_H, NM}, 128-byte swizzle.
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int make_proto_tmap(CUtensorMap *tm, const void *protos, int bf16, int B, int PH, int PW) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qr) != cudaSuccess || !sym ||
            qr != cudaDriverEntryPointSuccess)
            return BT_ERR_CUDA;
        fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    const cuuint64_t gdim[3] = {(cuuint64_t)PW, (cuuint64_t)PH, (cuuint64_t)B * NM};
    const cuuint64_t esz = bf16 ? 2 : 4;
    const cuuint64_t gstride[2] = {(cuuint64_t)PW * esz, (cuuint64_t)PW * PH * esz};
    const cuuint32_t box[3] = {(cuuint32_t)TA_W, (cuuint32_t)TA_H, (cuuint32_t)NM};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    // no L2 promotion (measured and not kept: 128 B / 256 B promotion, 48.0 / 50.5 us against 47.7 us without)
    const CUresult r = fn(tm, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void *>(protos),
                          gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          bf16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? BT_OK : BT_ERR_CUDA;
}

int launch_masks(const BtParams &p, const BtIO &io, const Workspace &w, cudaStream_t s, int parts) {
    K3Params P{};
    P.B = p.batch; P.S_h = p.img_h; P.S_w = p.img_w; P.PH = p.proto_h; P.PW = p.proto_w;
    P.K = p.max_det; P.gt_f32 = p.gt_mask_dtype == BT_MASK_F32;
    P.bias = p.proj_bias;
    P.protos = io.protos; P.proto_bf16 = p.proto_dtype == BT_PROTO_BF16; P.proj_weight = io.proj_weight; P.det_coeff = io.det_coeff;
    P.det_count = io.det_count; P.masks_gt = io.masks_gt; P.det_region = w.det_region; P.scr_off = w.scr_off;
    P.pool = w.pool; P.lm = w.lm; P.gtc = w.gtc; P.unc = w.unc; P.gpart = w.gpart;
    P.work = w.work; P.acc = w.acc; P.items = w.items; P.n_items = w.n_items; P.item_cap = (int)w.item_cap;
    P.tile_cnt = w.tile_cnt; P.tile_list = w.tile_list; P.inst_area = io.inst_area; P.inst_inter = io.inst_inter;
    P.seg_cnt4 = (long long *)io.seg_cnt4; P.uni_cnt4 = (long long *)io.uni_cnt4;
    P.seg_img3 = (long long *)io.seg_img3; P.uni_img3 = (long long *)io.uni_img3;
    P.seg_dice = io.seg_dice; P.seg_iou = io.seg_iou; P.uni_dice = io.uni_dice; P.uni_iou = io.uni_iou;
    P.seg_mask = io.seg_mask; P.uni_mask = io.uni_mask; P.seg_logits = io.seg_logits;
    P.seg_prob_sum = io.seg_prob_sum; P.sweep = static_cast<long long *>(io.sweep);
    P.inst_bits = reinterpret_cast<uint32_t *>(io.inst_bits); P.inst_masks = io.inst_masks;
    P.seg_sweep = static_cast<long long *>(io.seg_sweep); P.image_base = io.image_base; P.image_offset = p.image_offset;
    P.T = p.num_iou_thrs;
    for (int i = 0; i < p.num_iou_thrs; ++i) P.thrs[i] = p.iou_thrs[i];
    if (const BtIOSoftDice *sd = soft_io(p, io)) {
        P.seg_soft2 = reinterpret_cast<long long *>(sd->seg_soft2); P.seg_soft_dice = sd->seg_soft_dice;
        P.seg_soft_acc = reinterpret_cast<long long *>(sd->seg_soft_acc);
    }
    if (p.proto_w % (P.proto_bf16 ? 8 : 4) != 0) return BT_ERR_UNSUPPORTED;   // 16-byte global strides for the tensor map
    P.NBY = mask_blocks(p.proto_h); P.NBX = mask_blocks(p.proto_w);
    P.ntx = (p.proto_w + TA_W - 1) / TA_W; P.nty = (p.proto_h + TA_H - 1) / TA_H;
    P.m1_items = (P.NBY * P.NBX + 31) / 32;
    P.inv_K = 1.0f / (float)p.max_det; P.inv_m1 = 1.0f / (float)P.m1_items; P.inv_NBX = 1.0f / (float)P.NBX;
    {
        const int rows[3] = {0, P.NBY > 2 ? 1 : 0, P.NBY - 1}, cols[3] = {0, P.NBX > 2 ? 1 : 0, P.NBX - 1};
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) P.valid_tab[r * 3 + c] = block_valid_slow(rows[r], cols[c], p.proto_h, p.proto_w, p.img_h, p.img_w);
    }
    CUtensorMap tm;
    if (make_proto_tmap(&tm, io.protos, P.proto_bf16, p.batch, p.proto_h, p.proto_w) != BT_OK) return BT_ERR_CUDA;

    if (parts & BT_MASKS_PACK) {
        const size_t smem_g = (size_t)(8 * G_ROWS + 2) * (p.img_w / 32) * sizeof(uint32_t);
        gt_pack_kernel<<<dim3((P.NBY + G_ROWS - 1) / G_ROWS, p.batch), G_THREADS, smem_g, s>>>(P);
    }

    const size_t smem_a = (size_t)NM * TA_H * TA_W * (P.proto_bf16 ? 2 : 4) + 1024;
    // function attributes are per device: one flag per device ordinal
    static bool attr_done[64] = {};
    int attr_dev = 0;
    if (cudaGetDevice(&attr_dev) != cudaSuccess || attr_dev < 0 || attr_dev >= 64) return BT_ERR_CUDA;
    if (!attr_done[attr_dev]) {
        if (cudaFuncSetAttribute(contract_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(contract_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024) != cudaSuccess)
            return BT_ERR_CUDA;
        attr_done[attr_dev] = true;
    }
    {
        static int sm_count_dev[64] = {};   // per device ordinal, like the attribute flags above
        if (!sm_count_dev[attr_dev] &&
            (cudaDeviceGetAttribute(&sm_count_dev[attr_dev], cudaDevAttrMultiProcessorCount, attr_dev) != cudaSuccess ||
             sm_count_dev[attr_dev] <= 0))
            return BT_ERR_CUDA;
        const int sm_count = sm_count_dev[attr_dev];
        // BtParams.in_flight >= 2: several batches share the GPU.  Smaller grids of the two persistent kernels (3 / 6 CTAs per
        // SM instead of 4 / 8, which fill the register file) let the other batches' CTAs become resident beside them:
        // 93.1 -> 91.7 us per pipelined step (profiles/r02c_ctas.txt); alone, the kernels are fastest with the full grids.
        const bool shared_gpu = p.in_flight >= 2;
        const int ctas_per_sm_a = shared_gpu ? 3 : 4, ctas_per_sm_c = shared_gpu ? 6 : 8;   // contract_kernel, cells_kernel
        const int ntiles = p.batch * P.ntx * P.nty, cta_a = sm_count * ctas_per_sm_a;
        const int grid_a = ntiles < cta_a ? ntiles : cta_a;
        if (parts & BT_MASKS_CONTRACT) {
            if (P.proto_bf16) contract_kernel<true><<<grid_a, A_THREADS, smem_a, s>>>(P, tm);
            else contract_kernel<false><<<grid_a, A_THREADS, smem_a, s>>>(P, tm);
        }
        const long long items = (long long)p.batch * (p.max_det + P.m1_items);   // grid sizing only: the kernel reads the real count
        const long long want = (items + C_WARPS - 1) / C_WARPS, cap = (long long)sm_count * ctas_per_sm_c;
        if (parts & BT_MASKS_CELLS) {
            const long long ctas = want < cap ? want : cap;
            P.nq = 1;   // queues: a power of two <= warps in the grid (every queue needs a home warp), at most C_NQ
            while (P.nq * 2 <= C_NQ && P.nq * 2 <= ctas * C_WARPS) P.nq *= 2;
            const size_t inst_words = (size_t)p.batch * p.max_det * p.img_h * (p.img_w / 32);
            if (io.inst_bits && cudaMemsetAsync(io.inst_bits, 0, inst_words * 4, s) != cudaSuccess) return BT_ERR_CUDA;
            cells_kernel<<<(unsigned)ctas, C_WARPS * 32, 0, s>>>(P);
            if (io.inst_bits && io.inst_masks) {
                const size_t want_d = (inst_words + C_THREADS - 1) / C_THREADS, cap_d = (size_t)sm_count * 16;
                inst_dense_kernel<<<(unsigned)(want_d < cap_d ? want_d : cap_d), C_THREADS, 0, s>>>(P.inst_bits, io.inst_masks, inst_words);
            }
            finalize_kernel<<<(p.batch + C_THREADS / 32 - 1) / (C_THREADS / 32), C_THREADS, 0, s>>>(P);
            if (io.uni_mask) union_dense_kernel<<<p.batch, C_THREADS, 0, s>>>(P);
        }
    }
    return cudaGetLastError() == cudaSuccess ? BT_OK : BT_ERR_CUDA;
}

int launch_seg_curve(const BtParams &p, const Workspace &w, const float *thr, int T, int64_t *hist, cudaStream_t s) {
    CurveParams P{};
    P.B = p.batch; P.S_h = p.img_h; P.S_w = p.img_w; P.PH = p.proto_h; P.PW = p.proto_w;
    P.NBY = mask_blocks(p.proto_h); P.NBX = mask_blocks(p.proto_w);
    P.T = T; P.span = next_pow2(T + 1);
    P.lm = w.lm; P.gtc = w.gtc; P.hist = reinterpret_cast<unsigned long long *>(hist);
    for (int i = 0; i < T; ++i) P.thr[i] = thr[i];
    static int sm_count_dev[64] = {};   // per device ordinal, as in launch_masks
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return BT_ERR_CUDA;
    if (!sm_count_dev[dev] &&
        (cudaDeviceGetAttribute(&sm_count_dev[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sm_count_dev[dev] <= 0))
        return BT_ERR_CUDA;
    // A CTA's u32 bins count at most about 64 * blocks / grid pixels: the grid grows before that could reach 2^31.
    const long long blocks = (long long)p.batch * P.NBY * P.NBX;
    long long grid = (blocks + CV_THREADS - 1) / CV_THREADS, cap = (long long)sm_count_dev[dev] * CV_CTAS_PER_SM;
    if (grid > cap) grid = cap;
    const long long min_grid = (blocks * 64 + 0x7fffffffll) / 0x80000000ll;
    if (grid < min_grid) grid = min_grid;
    seg_curve_kernel<<<(unsigned)grid, CV_THREADS, 0, s>>>(P);
    return cudaGetLastError() == cudaSuccess ? BT_OK : BT_ERR_CUDA;
}

}  // namespace bt
