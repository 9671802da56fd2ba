// Sweep state + COCOeval.accumulate on the device (include/btpost.h "Sweep state").
//
// Reference statements replaced (paths under /root/reference/src): torchmetrics MeanAveragePrecision's per-image
// state lists (running_main_v2.py:884-892, evaluate_model.py:180-182) and its compute() -> pycocotools
// COCOeval.accumulate (running_main_v2.py:1017-1098, evaluate_model.py:291-319; SURVEY.md A.3).
//
// Records are appended by match_kernel (nms_match.cu).  btpost_sweep_accumulate:
//   1. stable LSD radix sort, 8 bits per pass, of the 32-byte records by (class, score desc, image, rank): the order
//      pycocotools obtains by concatenating the images in order and a mergesort on -score.  One warp owns a tile of
//      1024 consecutive records: per-warp digit histograms -> one exclusive scan over (digit, warp) -> every warp
//      scatters its tile in order (ranks inside a round of 32 from __match_any_sync), which keeps the sort stable.
//      Passes over bytes that are zero for every record (image index / rank bounds known to the caller) are skipped.
//   2. per (class, maxDet, area range, IoU threshold) -- a "combo" -- running tp / fp counts in three steps over
//      class-aligned chunks of 256 records: chunk sums, exclusive scan of the chunk sums, walk.  The walk needs no
//      second sort or envelope array: the interpolated precision at recall threshold r is the maximum of
//      tp / (tp + fp + eps) over the TRUE-POSITIVE positions whose recall reaches r (a position where fp grows never
//      beats the true positive before it, and the right-to-left running max of pycocotools is exactly that maximum),
//      so every true positive does one atomic max into the bin of the LAST recall threshold it reaches and a suffix
//      max over the 101 bins finishes the job.  Doubles throughout, same expressions as numpy.
//   3. optional (btpost_sweep_accumulate_ext): pycocotools' `scores` table, written by the walk at the one position that
//      first reaches each recall threshold.
#include "common.cuh"

namespace bt {

typedef unsigned long long u64;

constexpr int RS_THREADS = 256, RS_WARPS = RS_THREADS / 32;
constexpr int RS_ROUNDS = 32, RS_WTILE = 32 * RS_ROUNDS;   // records per warp tile
constexpr int ACC_CHUNK = 256, ACC_THREADS = 128;
constexpr int ACC_MAX_COMBOS = 4 * BT_NUM_AREA * BT_MAX_IOU_THRS, ACC_MAX_REC = 128;

// sort key, least significant byte first: rank (2 bytes), image (4), score_key (4), label (1)
__device__ __forceinline__ unsigned key_byte(const uint4 &k, int field) {
    // second half of a BtSweepRecord: x = score_key, y = image, z = rank | class_rank << 16, w = label | pad
    switch (field) {
        case 0: return k.z & 0xffu;
        case 1: return (k.z >> 8) & 0xffu;
        case 2: return k.y & 0xffu;
        case 3: return (k.y >> 8) & 0xffu;
        case 4: return (k.y >> 16) & 0xffu;
        case 5: return k.y >> 24;
        case 6: return k.x & 0xffu;
        case 7: return (k.x >> 8) & 0xffu;
        case 8: return (k.x >> 16) & 0xffu;
        case 9: return k.x >> 24;
        default: return k.w & 0xffu;
    }
}

__global__ void __launch_bounds__(RS_THREADS) radix_hist_kernel(const uint4 *__restrict__ rec, long long n, int field, int nw,
                                                                unsigned *__restrict__ ghist) {
    __shared__ unsigned s_h[RS_WARPS][256];
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
    const int w = blockIdx.x * RS_WARPS + wl;
    for (int i = lane; i < 256; i += 32) s_h[wl][i] = 0;
    __syncwarp();
    if (w < nw) {
        const long long base = (long long)w * RS_WTILE;
        for (int r = 0; r < RS_ROUNDS; ++r) {
            const long long i = base + r * 32 + lane;
            if (i < n) atomicAdd(&s_h[wl][key_byte(__ldg(rec + 2 * i + 1), field)], 1u);
        }
        __syncwarp();
        for (int i = lane; i < 256; i += 32) ghist[(size_t)i * nw + w] = s_h[wl][i];
    }
}

// Scan of the [256][nw] counters in two levels: block d turns the nw counters of digit d into exclusive prefixes inside
// the digit and leaves the digit's total in dtot[d]; the scatter kernel adds the digit bases (a 256-element scan every
// block does for itself).  (One block scanning all 256 * nw counters took 0.2-0.3 ms per pass at 1.6 M records: most of
// the accumulate.)
__global__ void __launch_bounds__(1024) radix_scan_digit_kernel(unsigned *__restrict__ h, int nw, unsigned *__restrict__ dtot) {
    __shared__ unsigned s_w[32];
    __shared__ unsigned s_carry;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    unsigned *row = h + (size_t)blockIdx.x * nw;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < nw; base += 1024) {
        const int i = base + tid;
        const unsigned v = i < nw ? row[i] : 0u;
        unsigned incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned u = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += u;
        }
        if (lane == 31) s_w[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            unsigned x = s_w[lane], xi = x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned u = __shfl_up_sync(0xffffffffu, xi, d);
                if (lane >= d) xi += u;
            }
            s_w[lane] = xi - x;   // exclusive over the warps
        }
        __syncthreads();
        const unsigned carry = s_carry;
        if (i < nw) row[i] = carry + s_w[wid] + incl - v;
        __syncthreads();
        if (tid == 1023) s_carry = carry + s_w[31] + incl;
        __syncthreads();
    }
    if (tid == 0) dtot[blockIdx.x] = s_carry;
}

__global__ void __launch_bounds__(RS_THREADS) radix_scatter_kernel(const uint4 *__restrict__ rec, uint4 *__restrict__ out, long long n,
                                                                   int field, int nw, const unsigned *__restrict__ ghist,
                                                                   const unsigned *__restrict__ dtot) {
    __shared__ unsigned s_off[RS_WARPS][256];
    __shared__ unsigned s_base[256], s_wt[RS_WARPS];
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
    const int w = blockIdx.x * RS_WARPS + wl;
    {   // digit bases: exclusive scan of the 256 digit totals (RS_THREADS == 256: one digit per thread)
        const unsigned v = dtot[threadIdx.x];
        unsigned incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned u = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += u;
        }
        if (lane == 31) s_wt[wl] = incl;
        __syncthreads();
        unsigned before = 0;
        for (int q = 0; q < wl; ++q) before += s_wt[q];
        s_base[threadIdx.x] = before + incl - v;
        __syncthreads();
    }
    if (w >= nw) return;
    for (int i = lane; i < 256; i += 32) s_off[wl][i] = ghist[(size_t)i * nw + w] + s_base[i];
    __syncwarp();
    const long long base = (long long)w * RS_WTILE;
    const unsigned lt = (1u << lane) - 1u;
    for (int r = 0; r < RS_ROUNDS; ++r) {
        const long long i = base + r * 32 + lane;
        const bool act = i < n;
        const unsigned amask = __ballot_sync(0xffffffffu, act);
        if (!amask) break;
        if (act) {
            const uint4 lo = __ldg(rec + 2 * i), hi = __ldg(rec + 2 * i + 1);
            const unsigned d = key_byte(hi, field);
            const unsigned peers = __match_any_sync(amask, d);
            const unsigned b0 = s_off[wl][d];
            __syncwarp(amask);
            if (lane == __ffs(peers) - 1) s_off[wl][d] = b0 + __popc(peers);
            __syncwarp(amask);
            const long long dst = (long long)b0 + __popc(peers & lt);
            out[2 * dst] = lo;
            out[2 * dst + 1] = hi;
        }
    }
}

__global__ void sweep_reset_kernel(long long *hdr, long long capacity) {
    hdr[threadIdx.x] = threadIdx.x == BT_SWEEP_CAPACITY ? capacity : 0;
}

// ---- accumulate --------------------------------------------------------------------------------------------------
struct AccParams {
    const BtSweepRecord *rec;
    long long n;
    int nc, T, M, R, ncombo;       // combo = (m * A + a) * T + t
    int max_dets[4];
    const double *rec_thrs;
    const long long *npig;         // [A][BT_MAX_CLASSES]
    long long *cls_start;          // [nc + 1] first record of each class in the sorted list
    uint2 *sums;                   // [chunks][ncombo] (tp, fp): per-chunk counts, then exclusive prefixes inside the class
    uint2 *totals;                 // [nc][ncombo]
    u64 *table;                    // [nc][ncombo][R] bit patterns of non-negative doubles
    double *precision, *recall;
    double *scores;                // optional [T][R][nc][A][M] (btpost_sweep_accumulate_ext)
    u64 *first_inc;                // [nc][4] first record of each (class, maxDet) sequence (only with `scores`)
};

// fp32 score of a record (inverse of desc_key; -0.0 comes back as +0.0)
__device__ __forceinline__ double key_score(unsigned key) {
    const unsigned asc = ~key;
    return (double)__uint_as_float((asc & 0x80000000u) ? (asc & 0x7fffffffu) : ~asc);
}

__global__ void class_bounds_kernel(const AccParams P) {
    const int c = threadIdx.x;
    if (c > P.nc) return;
    long long lo = 0, hi = P.n;   // first index with label >= c
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if ((int)P.rec[mid].label < c) lo = mid + 1; else hi = mid;
    }
    P.cls_start[c] = (c == P.nc) ? P.n : lo;
}

// chunk index -> (class, first record, records in the chunk); false past the last chunk
__device__ __forceinline__ bool chunk_of(const AccParams &P, int chunk, int &c, long long &r0, int &cnt, int &first_chunk) {
    int acc = 0;
    for (c = 0; c < P.nc; ++c) {
        const long long len = P.cls_start[c + 1] - P.cls_start[c];
        const int nch = (int)((len + ACC_CHUNK - 1) / ACC_CHUNK);
        if (chunk < acc + nch) {
            r0 = P.cls_start[c] + (long long)(chunk - acc) * ACC_CHUNK;
            cnt = (int)min((long long)ACC_CHUNK, P.cls_start[c + 1] - r0);
            first_chunk = acc;
            return true;
        }
        acc += nch;
    }
    return false;
}

template <bool WALK>
__global__ void __launch_bounds__(ACC_THREADS) acc_chunk_kernel(const AccParams P) {
    __shared__ u64 s_m[ACC_CHUNK], s_i[ACC_CHUNK];
    __shared__ unsigned short s_cr[ACC_CHUNK];
    __shared__ unsigned s_sk[ACC_CHUNK];
    int c, cnt, first;
    long long r0;
    if (!chunk_of(P, blockIdx.x, c, r0, cnt, first)) return;
    for (int i = threadIdx.x; i < cnt; i += ACC_THREADS) {
        const BtSweepRecord &r = P.rec[r0 + i];
        s_m[i] = r.matched; s_i[i] = r.ignored; s_cr[i] = r.class_rank; s_sk[i] = r.score_key;
    }
    __syncthreads();
    const int A = BT_NUM_AREA;
    // score table: where each (class, maxDet) sequence starts -- its first record may be ignored at every (area,
    // threshold), so the tp / fp prefixes cannot tell the walk whether a chunk holds it
    if (!WALK && P.scores && threadIdx.x < P.M) {
        const int md = P.max_dets[threadIdx.x];
        for (int i = 0; i < cnt; ++i)
            if (s_cr[i] < md) { atomicMin(P.first_inc + c * 4 + threadIdx.x, (u64)(r0 + i)); break; }
    }
    for (int combo = threadIdx.x; combo < P.ncombo; combo += ACC_THREADS) {
        const int m = combo / (A * P.T), bit = combo - m * A * P.T, a = bit / P.T;
        const int md = P.max_dets[m];
        uint2 *slot = P.sums + (size_t)blockIdx.x * P.ncombo + combo;
        if (!WALK) {
            unsigned tp = 0, fp = 0;
            for (int i = 0; i < cnt; ++i) {
                const unsigned ok = (s_cr[i] < md) & (unsigned)(~(s_i[i] >> bit) & 1ull);
                const unsigned mt = (unsigned)((s_m[i] >> bit) & 1ull);
                tp += ok & mt;
                fp += ok & (mt ^ 1u);
            }
            *slot = make_uint2(tp, fp);
        } else {
            const long long npig = P.npig[a * BT_MAX_CLASSES + c];
            if (npig == 0) continue;
            const uint2 pre = *slot;
            unsigned tp = pre.x, fp = pre.y;
            const double npd = (double)npig, eps = 2.220446049250313e-16;   // numpy.spacing(1)
            u64 *tab = P.table + ((size_t)c * P.ncombo + combo) * P.R;
            int bin = -1, cur_bin = -1;
            double cur_max = 0.0;
            // score table: recall threshold r is first reached at the sequence's first record (r with rec_thrs[r] <= 0)
            // or at a true positive, and exactly one position reaches it first, so plain stores suffice.  sbin = last
            // threshold reached before the current position.
            double *sc = nullptr;
            size_t sc_stride = 0;
            u64 seq0 = ~0ull;
            int sbin = -1;
            if (P.scores) {
                const int t = bit - a * P.T;
                sc = P.scores + (((size_t)t * P.R * P.nc + c) * A + a) * P.M + m;
                sc_stride = (size_t)P.nc * A * P.M;
                seq0 = P.first_inc[c * 4 + m];
                if ((u64)r0 > seq0) {
                    const double rc0 = (double)tp / npd;
                    while (sbin + 1 < P.R && P.rec_thrs[sbin + 1] <= rc0) ++sbin;
                }
            }
            auto settle = [&](int i, double rc) {
                while (sbin + 1 < P.R && P.rec_thrs[sbin + 1] <= rc) sc[(size_t)(++sbin) * sc_stride] = key_score(s_sk[i]);
            };
            for (int i = 0; i < cnt; ++i) {
                const unsigned ok = (s_cr[i] < md) & (unsigned)(~(s_i[i] >> bit) & 1ull);
                if (!ok || !((s_m[i] >> bit) & 1ull)) {
                    fp += ok;
                    if (sc && (u64)(r0 + i) == seq0) settle(i, (double)tp / npd);
                    continue;
                }
                ++tp;
                const double rc = (double)tp / npd;
                if (sc) settle(i, rc);
                while (bin + 1 < P.R && P.rec_thrs[bin + 1] <= rc) ++bin;   // last recall threshold this position reaches
                if (bin < 0) continue;
                const double pr = (double)tp / ((double)(fp + tp) + eps);
                if (bin != cur_bin) {
                    if (cur_bin >= 0) atomicMax(tab + cur_bin, (u64)__double_as_longlong(cur_max));
                    cur_bin = bin; cur_max = pr;
                } else if (pr > cur_max) {
                    cur_max = pr;
                }
            }
            if (cur_bin >= 0) atomicMax(tab + cur_bin, (u64)__double_as_longlong(cur_max));
        }
    }
}

// exclusive scan of the chunk sums inside every class, one warp per (combo, class)
__global__ void __launch_bounds__(32) acc_scan_kernel(const AccParams P) {
    const int combo = blockIdx.x, c = blockIdx.y, lane = threadIdx.x;
    int first = 0;
    for (int q = 0; q < c; ++q) first += (int)((P.cls_start[q + 1] - P.cls_start[q] + ACC_CHUNK - 1) / ACC_CHUNK);
    const int nch = (int)((P.cls_start[c + 1] - P.cls_start[c] + ACC_CHUNK - 1) / ACC_CHUNK);
    unsigned ctp = 0, cfp = 0;
    for (int j0 = 0; j0 < nch; j0 += 32) {
        const int j = j0 + lane;
        uint2 v = make_uint2(0, 0);
        if (j < nch) v = P.sums[(size_t)(first + j) * P.ncombo + combo];
        unsigned itp = v.x, ifp = v.y;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned a = __shfl_up_sync(0xffffffffu, itp, d), b = __shfl_up_sync(0xffffffffu, ifp, d);
            if (lane >= d) { itp += a; ifp += b; }
        }
        if (j < nch) P.sums[(size_t)(first + j) * P.ncombo + combo] = make_uint2(ctp + itp - v.x, cfp + ifp - v.y);
        ctp += __shfl_sync(0xffffffffu, itp, 31);
        cfp += __shfl_sync(0xffffffffu, ifp, 31);
    }
    if (lane == 0) P.totals[(size_t)c * P.ncombo + combo] = make_uint2(ctp, cfp);
    if (P.scores) {   // the walk overwrites the thresholds that some record reaches
        const int A = BT_NUM_AREA, m = combo / (A * P.T), bit = combo - m * A * P.T, a = bit / P.T, t = bit - a * P.T;
        const double v = P.npig[a * BT_MAX_CLASSES + c] == 0 ? -1.0 : 0.0;
        for (int r = lane; r < P.R; r += 32) P.scores[((((size_t)t * P.R + r) * P.nc + c) * A + a) * P.M + m] = v;
    }
}

__global__ void __launch_bounds__(ACC_THREADS) acc_final_kernel(const AccParams P) {
    const int A = BT_NUM_AREA;
    const int idx = blockIdx.x * ACC_THREADS + threadIdx.x;
    if (idx >= P.nc * P.ncombo) return;
    const int c = idx / P.ncombo, combo = idx - c * P.ncombo;
    const int m = combo / (A * P.T), bit = combo - m * A * P.T, a = bit / P.T, t = bit - a * P.T;
    const long long npig = P.npig[a * BT_MAX_CLASSES + c];
    const u64 *tab = P.table + ((size_t)c * P.ncombo + combo) * P.R;
    double run = 0.0;
    for (int r = P.R - 1; r >= 0; --r) {
        double v = -1.0;
        if (npig != 0) {
            run = fmax(run, __longlong_as_double((long long)tab[r]));
            v = run;
        }
        P.precision[((((size_t)t * P.R + r) * P.nc + c) * A + a) * P.M + m] = v;
    }
    P.recall[(((size_t)t * P.nc + c) * A + a) * P.M + m] =
        npig != 0 ? (double)P.totals[(size_t)c * P.ncombo + combo].x / (double)npig : -1.0;
}

struct AccScratch {
    uint4 *tmp;           // second record buffer of the radix sort
    unsigned *ghist;      // [256][warps]
    unsigned *dtot;       // [256] records per digit
    long long *cls_start;
    uint2 *sums, *totals;
    u64 *table;
    u64 *first_inc;       // [BT_MAX_CLASSES][4]
    size_t bytes;
};
static AccScratch acc_carve(long long n, void *base) {
    AccScratch s;
    char *ptr = static_cast<char *>(base);
    size_t off = 0;
    auto take = [&](size_t b) {
        char *r = ptr ? ptr + off : nullptr;
        off += align_up(b, 256);
        return r;
    };
    const long long nw = (n + RS_WTILE - 1) / RS_WTILE;
    const long long chunks = (n + ACC_CHUNK - 1) / ACC_CHUNK + BT_MAX_CLASSES;
    s.tmp = reinterpret_cast<uint4 *>(take((size_t)(n > 0 ? n : 1) * sizeof(BtSweepRecord)));
    s.ghist = reinterpret_cast<unsigned *>(take((size_t)256 * (nw > 0 ? nw : 1) * sizeof(unsigned)));
    s.dtot = reinterpret_cast<unsigned *>(take(256 * sizeof(unsigned)));
    s.cls_start = reinterpret_cast<long long *>(take((BT_MAX_CLASSES + 1) * sizeof(long long)));
    s.sums = reinterpret_cast<uint2 *>(take((size_t)chunks * ACC_MAX_COMBOS * sizeof(uint2)));
    s.totals = reinterpret_cast<uint2 *>(take((size_t)BT_MAX_CLASSES * ACC_MAX_COMBOS * sizeof(uint2)));
    s.table = reinterpret_cast<u64 *>(take((size_t)BT_MAX_CLASSES * ACC_MAX_COMBOS * ACC_MAX_REC * sizeof(u64)));
    s.first_inc = reinterpret_cast<u64 *>(take((size_t)BT_MAX_CLASSES * 4 * sizeof(u64)));
    s.bytes = off;
    return s;
}

}  // namespace bt

using namespace bt;

extern "C" {

int btpost_sweep_bytes(int64_t max_records, size_t *bytes) {
    if (!bytes || max_records < 0) return BT_ERR_BAD_ARG;
    *bytes = (size_t)BT_SWEEP_HEADER_I64 * 8 + (size_t)max_records * sizeof(BtSweepRecord);
    return BT_OK;
}

int btpost_sweep_reset(void *sweep, int64_t max_records, void *stream) {
    if (!sweep || max_records < 0) return BT_ERR_BAD_ARG;
    if (reinterpret_cast<uintptr_t>(sweep) & 15) return BT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    sweep_reset_kernel<<<1, BT_SWEEP_HEADER_I64, 0, s>>>(static_cast<long long *>(sweep), (long long)max_records);
    return cudaGetLastError() == cudaSuccess ? BT_OK : BT_ERR_CUDA;
}

int btpost_sweep_accumulate_bytes(int64_t n_records, size_t *bytes) {
    if (!bytes || n_records < 0) return BT_ERR_BAD_ARG;
    *bytes = acc_carve(n_records, nullptr).bytes;
    return BT_OK;
}

int btpost_sweep_accumulate(void *records, int64_t n_records, const int64_t *npig, const double *rec_thrs, int32_t num_rec,
                            int32_t nc, int32_t num_iou_thrs, const int32_t *max_dets, int32_t num_max_dets,
                            int32_t max_det_per_image, int64_t num_images, double *precision, double *recall, void *scratch,
                            size_t scratch_bytes, void *stream) {
    return btpost_sweep_accumulate_ext(records, n_records, npig, rec_thrs, num_rec, nc, num_iou_thrs, max_dets, num_max_dets,
                                       max_det_per_image, num_images, precision, recall, nullptr, scratch, scratch_bytes, stream);
}

int btpost_sweep_accumulate_ext(void *records, int64_t n_records, const int64_t *npig, const double *rec_thrs, int32_t num_rec,
                                int32_t nc, int32_t num_iou_thrs, const int32_t *max_dets, int32_t num_max_dets,
                                int32_t max_det_per_image, int64_t num_images, double *precision, double *recall,
                                double *scores, void *scratch, size_t scratch_bytes, void *stream) {
    if (!npig || !rec_thrs || !max_dets || !precision || !recall || !scratch || n_records < 0 || (n_records > 0 && !records))
        return BT_ERR_BAD_ARG;
    if (nc <= 0 || nc > BT_MAX_CLASSES || num_iou_thrs <= 0 || num_iou_thrs > BT_MAX_IOU_THRS || num_max_dets <= 0 ||
        num_max_dets > 4 || num_rec <= 0 || num_rec > ACC_MAX_REC || max_det_per_image <= 0 || num_images < 0)
        return BT_ERR_BAD_ARG;
    if ((reinterpret_cast<uintptr_t>(scratch) & 255) || (reinterpret_cast<uintptr_t>(records) & 15)) return BT_ERR_MISALIGNED;
    const AccScratch sc = acc_carve(n_records, scratch);
    if (scratch_bytes < sc.bytes) return BT_ERR_WORKSPACE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const long long n = n_records;
    const uint4 *src = static_cast<const uint4 *>(records);
    if (n > 0) {
        // ---- 1. radix sort; bytes that are zero everywhere are skipped
        const int nw = (int)((n + RS_WTILE - 1) / RS_WTILE), blocks = (nw + RS_WARPS - 1) / RS_WARPS;
        bool need[11];
        need[0] = true; need[1] = max_det_per_image > 256;
        for (int k = 0; k < 4; ++k) need[2 + k] = k == 0 || (num_images - 1) >> (8 * k) != 0;
        for (int k = 0; k < 4; ++k) need[6 + k] = true;
        need[10] = nc > 1;
        uint4 *bufs[2] = {static_cast<uint4 *>(records), sc.tmp};
        int cur = 0;
        for (int f = 0; f < 11; ++f) {
            if (!need[f]) continue;
            radix_hist_kernel<<<blocks, RS_THREADS, 0, s>>>(bufs[cur], n, f, nw, sc.ghist);
            radix_scan_digit_kernel<<<256, 1024, 0, s>>>(sc.ghist, nw, sc.dtot);
            radix_scatter_kernel<<<blocks, RS_THREADS, 0, s>>>(bufs[cur], bufs[cur ^ 1], n, f, nw, sc.ghist, sc.dtot);
            cur ^= 1;
        }
        if (cur == 1 && cudaMemcpyAsync(records, sc.tmp, (size_t)n * sizeof(BtSweepRecord), cudaMemcpyDeviceToDevice, s) != cudaSuccess)
            return BT_ERR_CUDA;
        src = static_cast<const uint4 *>(records);
    }
    // ---- 2. tp / fp scans and the interpolated precision
    AccParams P{};
    P.rec = reinterpret_cast<const BtSweepRecord *>(src);
    P.n = n; P.nc = nc; P.T = num_iou_thrs; P.M = num_max_dets; P.R = num_rec;
    P.ncombo = num_max_dets * BT_NUM_AREA * num_iou_thrs;
    for (int i = 0; i < num_max_dets; ++i) P.max_dets[i] = max_dets[i];
    P.rec_thrs = rec_thrs; P.npig = reinterpret_cast<const long long *>(npig);
    P.cls_start = sc.cls_start; P.sums = sc.sums; P.totals = sc.totals; P.table = sc.table;
    P.precision = precision; P.recall = recall;
    P.scores = scores; P.first_inc = sc.first_inc;
    if (cudaMemsetAsync(sc.table, 0, (size_t)nc * P.ncombo * num_rec * sizeof(u64), s) != cudaSuccess) return BT_ERR_CUDA;
    if (scores && cudaMemsetAsync(sc.first_inc, 0xff, (size_t)BT_MAX_CLASSES * 4 * sizeof(u64), s) != cudaSuccess) return BT_ERR_CUDA;
    class_bounds_kernel<<<1, 32, 0, s>>>(P);
    const int chunks = (int)((n + ACC_CHUNK - 1) / ACC_CHUNK) + nc;
    acc_chunk_kernel<false><<<chunks, ACC_THREADS, 0, s>>>(P);
    acc_scan_kernel<<<dim3(P.ncombo, nc), 32, 0, s>>>(P);
    acc_chunk_kernel<true><<<chunks, ACC_THREADS, 0, s>>>(P);
    acc_final_kernel<<<(nc * P.ncombo + ACC_THREADS - 1) / ACC_THREADS, ACC_THREADS, 0, s>>>(P);
    return cudaGetLastError() == cudaSuccess ? BT_OK : BT_ERR_CUDA;
}

}  // extern "C"
