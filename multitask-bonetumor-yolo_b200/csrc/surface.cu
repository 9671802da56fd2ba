// Surface distances of the projector mask against the GT mask (btpost_surface_distance): Hausdorff distance, HD95 and
// ASSD per image, MONAI's compute_hausdorff_distance / compute_average_surface_distance made exact (DESIGN.md §4).
//
// Per image, on integer squared distances only:
//   1. surface_cols_kernel: the edge pixels of P and of G (M AND NOT erode(M), 4-neighbour cross, background outside
//      the image), then per column the vertical distance to the nearest edge pixel of that column (two scans).
//   2. surface_rows_kernel: per row, the lower envelope of the parabolas (x - c)^2 + g(c)^2 over the columns c
//      (Felzenszwalb-Huttenlocher, intersections compared exactly in int64), evaluated at the other mask's edge pixels:
//      the exact squared Euclidean distance to the nearest edge pixel, written back in place, flagged.
//   3. surface_stats_kernel: per (image, direction) the count, the largest value, the sum of the distances in 2^-30
//      fixed point and the two order statistics of the 0.95 quantile (two-level histogram select on the 22-bit values).
//   4. surface_finish_kernel: HD, HD95 and ASSD per image, and the accumulator words.
// Everything is a pure function of the two masks: no atomics on floating-point values, so the bytes do not depend on the
// launch configuration or on the other images of the batch.
#include <math.h>

#include "common.cuh"

namespace bt {
namespace {

constexpr int SD_MAX_IMG = 1280;
constexpr uint32_t SD_FLAG = 0x80000000u;   // plane entry of an edge pixel: FLAG | squared distance (< 2^22)
constexpr uint32_t SD_D2_MASK = (1u << 22) - 1;
constexpr uint32_t SD_INF = 0xFFFFu;        // column distance in a column without edge pixels
constexpr int COL_THREADS = 128;
constexpr int ROW_THREADS = 32;             // rows per block; each thread keeps an envelope stack of S uint16 in shared memory
constexpr int STAT_THREADS = 512;
constexpr int SEL_BITS = 11;                // two-level select: 2048 bins of the high 11 bits, then of the low 11 bits
constexpr int SEL_BINS = 1 << SEL_BITS;
constexpr double SD_FX = 1073741824.0;      // 2^30: fixed point of the per-pixel distance terms of the ASSD sum
constexpr double SD_ACC = 4294967296.0;     // 2^32: fixed point of the accumulator words

struct SurfStat {            // one (image, direction)
    long long n;             // edge pixels of the query mask (0 when either mask is empty)
    long long sum;           // sum of round(sqrt(d2) * 2^30)
    unsigned int max2;       // largest squared distance
    unsigned int pad;
    double q95;              // torch.quantile(distances, 0.95)
};
static_assert(sizeof(SurfStat) == 32, "SurfStat layout");

size_t planes_bytes(int B, int S) { return (size_t)B * 2 * S * S * sizeof(uint32_t); }
size_t scratch_bytes(int B, int S) { return planes_bytes(B, S) + (((size_t)B * 2 * sizeof(SurfStat) + 255) & ~(size_t)255); }

template <typename GT>
__global__ void __launch_bounds__(COL_THREADS) surface_cols_kernel(const uint8_t *__restrict__ pred, const GT *__restrict__ gt,
                                                                   uint32_t *__restrict__ planes, int S) {
    const int x = blockIdx.x * COL_THREADS + threadIdx.x;
    const int m = blockIdx.y & 1, b = blockIdx.y >> 1;   // plane m: 0 = P (projector mask), 1 = G (GT mask)
    if (x >= S) return;
    const size_t img = (size_t)b * S * S;
    uint32_t *g = planes + ((size_t)b * 2 + m) * S * S;
    auto in = [&](int y, int xx) -> bool {
        if (y < 0 || y >= S || xx < 0 || xx >= S) return false;   // outside the image is background
        const size_t i = img + (size_t)y * S + xx;
        return m == 0 ? pred[i] != 0 : gt[i] != GT(0);
    };
    // downward scan: distance to the nearest edge pixel above (or at) y in this column
    bool up = false, cur = in(0, x);
    uint32_t d = SD_INF;
    for (int y = 0; y < S; ++y) {
        const bool down = in(y + 1, x);
        const bool edge = cur && !(up && down && in(y, x - 1) && in(y, x + 1));
        d = edge ? 0u : (d == SD_INF ? SD_INF : d + 1);
        g[(size_t)y * S + x] = d;
        up = cur;
        cur = down;
    }
    // upward scan: the nearest edge pixel below
    d = SD_INF;
    for (int y = S - 1; y >= 0; --y) {
        const uint32_t v = g[(size_t)y * S + x];
        d = v == 0 ? 0u : (d == SD_INF ? SD_INF : d + 1);
        if (d < v) g[(size_t)y * S + x] = d;
    }
}

// Column distance of a target-plane entry: an edge pixel (0, or flagged by an earlier pass) is 0; -1 = no edge pixel in the column.
__device__ __forceinline__ long long col_dist(uint32_t v) { return (v & SD_FLAG) ? 0 : v == SD_INF ? -1 : (long long)v; }

// One row, one direction: squared distance from every edge pixel of the query row (entry 0) to the nearest edge pixel of
// the target mask, written into the query row as FLAG | d2.  `stk` = this thread's stack (stride ROW_THREADS).
__device__ void envelope_row(const uint32_t *tgt, uint32_t *qry, uint16_t *stk, int S) {
    int top = -1;
    for (int c = 0; c < S; ++c) {
        const long long fc = col_dist(tgt[c]);
        if (fc < 0) continue;
        const long long hc = fc * fc + (long long)c * c;
        // pop the top parabola b while its intersection with c lies at or left of its intersection with the one below it
        while (top >= 1) {
            const int a = stk[(top - 1) * ROW_THREADS], bb = stk[top * ROW_THREADS];
            const long long fa = col_dist(tgt[a]), fb = col_dist(tgt[bb]);
            const long long ha = fa * fa + (long long)a * a, hb = fb * fb + (long long)bb * bb;
            // x(b, c) <= x(a, b) with x(u, v) = (h_v - h_u) / (2 (v - u))
            if ((hc - hb) * (bb - a) <= (hb - ha) * (c - bb)) --top;
            else break;
        }
        stk[++top * ROW_THREADS] = (uint16_t)c;
    }
    if (top < 0) return;   // the target mask is empty: the image is undefined, nothing is flagged
    int k = 0;
    long long fk = col_dist(tgt[stk[0]]);
    for (int x = 0; x < S; ++x) {
        if (qry[x] != 0) continue;   // not an edge pixel of the query mask
        long long best = (long long)(x - stk[k * ROW_THREADS]) * (x - stk[k * ROW_THREADS]) + fk * fk;
        while (k < top) {            // the envelope's pieces are ordered: move right while the next one is not above
            const int c1 = stk[(k + 1) * ROW_THREADS];
            const long long f1 = col_dist(tgt[c1]);
            const long long v1 = (long long)(x - c1) * (x - c1) + f1 * f1;
            if (v1 > best) break;
            ++k;
            fk = f1;
            best = v1;
        }
        qry[x] = SD_FLAG | (uint32_t)best;
    }
}

__global__ void __launch_bounds__(ROW_THREADS) surface_rows_kernel(uint32_t *__restrict__ planes, int B, int S) {
    extern __shared__ uint16_t s_stack[];
    const int r = blockIdx.x * ROW_THREADS + threadIdx.x;
    if (r >= B * S) return;
    const int b = r / S, y = r - b * S;
    uint32_t *p_row = planes + ((size_t)b * 2 + 0) * S * S + (size_t)y * S;
    uint32_t *g_row = planes + ((size_t)b * 2 + 1) * S * S + (size_t)y * S;
    uint16_t *stk = s_stack + threadIdx.x;
    // G -> P first: it reads the P row as the target and flags the G row's edge pixels, whose column distance (0) the
    // P -> G pass then reads back through col_dist.  One thread owns both rows of a row index, so this is race-free.
    envelope_row(p_row, g_row, stk, S);
    envelope_row(g_row, p_row, stk, S);
}

// Bin of the element of 0-based rank r in a SEL_BINS histogram and the number of elements in the bins before it
// (one thread writes them).  Every thread of the block calls it.
__device__ void select_bin(const unsigned int *h, long long r, int *bin, long long *below, long long *s_warp) {
    static_assert(SEL_BINS == 4 * STAT_THREADS, "four bins per thread");
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    unsigned int c[4];
    long long loc = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) { c[j] = h[4 * tid + j]; loc += c[j]; }
    long long inc = loc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[w] = inc;
    __syncthreads();
    long long run = inc - loc;
    for (int i = 0; i < w; ++i) run += s_warp[i];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (r >= run && r < run + c[j]) { *bin = 4 * tid + j; *below = run; }
        run += c[j];
    }
    __syncthreads();
}

// Histogram increment with the lanes of a warp that share a bin folded into one shared-memory atomic (most distances
// fall into a few bins).  All 32 lanes call it; `key` < 0 adds nothing.
__device__ __forceinline__ void warp_hist_add(unsigned int *h, int key) {
    const unsigned int peers = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&h[key], __popc(peers));
}

__global__ void __launch_bounds__(STAT_THREADS) surface_stats_kernel(const uint32_t *__restrict__ planes, SurfStat *__restrict__ st, int S) {
    __shared__ unsigned int h1[SEL_BINS], h2[2][SEL_BINS];
    __shared__ long long s_warp[STAT_THREADS / 32], s_n[STAT_THREADS / 32], s_sum[STAT_THREADS / 32];
    __shared__ unsigned int s_max[STAT_THREADS / 32];
    __shared__ int s_bin[2];
    __shared__ long long s_below[2];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const uint4 *pl = reinterpret_cast<const uint4 *>(planes + (size_t)blockIdx.x * S * S);   // plane 2b + dir
    const int n4 = S * S / 4;   // a multiple of 32 (S % 32 == 0): a warp's lanes run the same iterations (warp_hist_add)
    for (int i = tid; i < SEL_BINS; i += STAT_THREADS) h1[i] = h2[0][i] = h2[1][i] = 0;
    __syncthreads();
    long long n = 0, sum = 0;
    unsigned int mx = 0;
    for (int i = tid; i < n4; i += STAT_THREADS) {
        const uint4 v4 = pl[i];
        const uint32_t vs[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t v = vs[j];
            int key = -1;
            if (v & SD_FLAG) {
                const uint32_t d2 = v & SD_D2_MASK;
                ++n;
                sum += __double2ll_rn(__dmul_rn(__dsqrt_rn((double)d2), SD_FX));
                mx = max(mx, d2);
                key = (int)(d2 >> SEL_BITS);
            }
            warp_hist_add(h1, key);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n += __shfl_xor_sync(0xffffffffu, n, o);
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) { s_n[w] = n; s_sum[w] = sum; s_max[w] = mx; }
    __syncthreads();
    n = sum = 0;
    mx = 0;
    for (int i = 0; i < STAT_THREADS / 32; ++i) { n += s_n[i]; sum += s_sum[i]; mx = max(mx, s_max[i]); }
    if (n == 0) {
        if (tid == 0) st[blockIdx.x] = SurfStat{0, 0, 0, 0, 0.0};
        return;
    }
    // torch.quantile(x, 0.95), linear: rank = 0.95 (n - 1), the floor and ceil order statistics, lerp
    const double rank = __dmul_rn(0.95, (double)(n - 1));
    const long long r_lo = (long long)floor(rank), r_hi = (long long)ceil(rank);
    select_bin(h1, r_lo, &s_bin[0], &s_below[0], s_warp);
    select_bin(h1, r_hi, &s_bin[1], &s_below[1], s_warp);
    const int bin_lo = s_bin[0], bin_hi = s_bin[1];
    for (int i = tid; i < n4; i += STAT_THREADS) {
        const uint4 v4 = pl[i];
        const uint32_t vs[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t v = vs[j];
            const int hb = (v & SD_FLAG) ? (int)((v & SD_D2_MASK) >> SEL_BITS) : -1;
            const int low = (int)(v & (SEL_BINS - 1));
            warp_hist_add(h2[0], hb == bin_lo ? low : -1);
            if (bin_hi != bin_lo) warp_hist_add(h2[1], hb == bin_hi ? low : -1);
        }
    }
    __syncthreads();
    const long long below_lo = s_below[0], below_hi = s_below[1];
    select_bin(h2[0], r_lo - below_lo, &s_bin[0], &s_below[0], s_warp);
    select_bin(h2[bin_hi != bin_lo ? 1 : 0], r_hi - below_hi, &s_bin[1], &s_below[1], s_warp);
    if (tid == 0) {
        const double a = __dsqrt_rn((double)(((uint32_t)bin_lo << SEL_BITS) | (uint32_t)s_bin[0]));
        const double bv = __dsqrt_rn((double)(((uint32_t)bin_hi << SEL_BITS) | (uint32_t)s_bin[1]));
        const double wgt = __dsub_rn(rank, (double)r_lo);
        const double diff = __dsub_rn(bv, a);
        const double q = wgt < 0.5 ? __dadd_rn(a, __dmul_rn(wgt, diff)) : __dsub_rn(bv, __dmul_rn(diff, __dsub_rn(1.0, wgt)));
        st[blockIdx.x] = SurfStat{n, sum, mx, 0, q};
    }
}

__global__ void surface_finish_kernel(const SurfStat *__restrict__ st, int B, float *hd, float *hd95, float *assd, int64_t *acc) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const SurfStat P = st[2 * b], G = st[2 * b + 1];
    if (P.n == 0 || G.n == 0) {   // either mask empty: undefined, not counted
        hd[b] = hd95[b] = assd[b] = __int_as_float(0x7fc00000);
        return;
    }
    const float h = __double2float_rn(__dsqrt_rn((double)max(P.max2, G.max2)));
    const float h95 = __double2float_rn(fmax(P.q95, G.q95));
    const float as = __double2float_rn(__ddiv_rn(__ddiv_rn((double)(P.sum + G.sum), SD_FX), (double)(P.n + G.n)));
    hd[b] = h;
    hd95[b] = h95;
    assd[b] = as;
    if (acc) {
        auto add = [](int64_t *p, long long v) { atomicAdd(reinterpret_cast<unsigned long long *>(p), (unsigned long long)v); };
        add(acc + 0, __double2ll_rn(__dmul_rn((double)h, SD_ACC)));
        add(acc + 1, __double2ll_rn(__dmul_rn((double)h95, SD_ACC)));
        add(acc + 2, __double2ll_rn(__dmul_rn((double)as, SD_ACC)));
        add(acc + 3, 1);
    }
}

}  // namespace
}  // namespace bt

using namespace bt;

extern "C" {

int btpost_surface_bytes(int32_t batch, int32_t img, size_t *bytes) {
    if (!bytes || batch <= 0 || img <= 0) return BT_ERR_BAD_ARG;
    if (img % 32 != 0 || img > SD_MAX_IMG) return BT_ERR_UNSUPPORTED;
    *bytes = scratch_bytes(batch, img);
    return BT_OK;
}

int btpost_surface_distance(int32_t batch, int32_t img, const uint8_t *pred, const void *gt, int32_t gt_mask_dtype, float *hd,
                            float *hd95, float *assd, int64_t *acc, void *scratch, size_t scratch_bytes_, void *stream) {
    if (!pred || !gt || !hd || !hd95 || !assd || !scratch || batch <= 0 || img <= 0) return BT_ERR_BAD_ARG;
    if (gt_mask_dtype != BT_MASK_U8 && gt_mask_dtype != BT_MASK_F32) return BT_ERR_BAD_ARG;
    if (img % 32 != 0 || img > SD_MAX_IMG) return BT_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(pred) & 15) || (reinterpret_cast<uintptr_t>(gt) & 15)) return BT_ERR_MISALIGNED;
    if (reinterpret_cast<uintptr_t>(scratch) & 255) return BT_ERR_MISALIGNED;
    if (scratch_bytes_ < scratch_bytes(batch, img)) return BT_ERR_WORKSPACE;
    const int B = batch, S = img;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint32_t *planes = static_cast<uint32_t *>(scratch);
    SurfStat *st = reinterpret_cast<SurfStat *>(static_cast<char *>(scratch) + planes_bytes(B, S));
    const size_t smem_rows = (size_t)ROW_THREADS * S * sizeof(uint16_t);
    static bool attr_done[64] = {};   // function attributes are per device: one flag per device ordinal
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return BT_ERR_CUDA;
    if (!attr_done[dev]) {
        if (cudaFuncSetAttribute(surface_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(ROW_THREADS * SD_MAX_IMG * sizeof(uint16_t))) != cudaSuccess)
            return BT_ERR_CUDA;
        attr_done[dev] = true;
    }
    const dim3 gcols((S + COL_THREADS - 1) / COL_THREADS, 2 * B);
    if (gt_mask_dtype == BT_MASK_U8)
        surface_cols_kernel<uint8_t><<<gcols, COL_THREADS, 0, s>>>(pred, static_cast<const uint8_t *>(gt), planes, S);
    else
        surface_cols_kernel<float><<<gcols, COL_THREADS, 0, s>>>(pred, static_cast<const float *>(gt), planes, S);
    surface_rows_kernel<<<(B * S + ROW_THREADS - 1) / ROW_THREADS, ROW_THREADS, smem_rows, s>>>(planes, B, S);
    surface_stats_kernel<<<2 * B, STAT_THREADS, 0, s>>>(planes, st, S);
    surface_finish_kernel<<<(B + 127) / 128, 128, 0, s>>>(st, B, hd, hd95, assd, acc);
    return cudaGetLastError() == cudaSuccess ? BT_OK : BT_ERR_CUDA;
}

}  // extern "C"
