// Multi-person pose AP (poseval's assignGTmulti + computeMetrics) over the packed parse result, sm_100a.
//
// The specification is the float64 restatement documented in DESIGN.md §12.  Two stages:
//   ap_match_kernel    one CTA per image: PCKh distances of every (prediction, GT person, joint), the two arg-max
//                      passes of assignGTmulti, and per (slot, joint) the entry's score and TP label.  Everything the
//                      second stage needs is copied out, so the parser's buffers may be reused for the next batch.
//   finalize           once per pass: compaction of the used slots into one 64-bit key per entry, a CUB segmented
//                      radix sort per joint, and one CTA per joint for the precision / recall curve and VOCap.
// Built with the library's flags (-fmad=false, IEEE division and square root); the fp64 distances are written with
// the __d*_rn intrinsics on top of that, one rounding per operation.
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>

#include "ppn_kernels.h"

namespace ppn {

namespace {

constexpr int kMatchThreads = 256;          // 8 warps, one prediction per warp at a time, lane = joint
constexpr int kCurveThreads = 512;
constexpr int kCurveItems = 8;              // entries per thread per tile of the curve scan
constexpr int kScanThreads = 1024;
constexpr int kKeyThreads = 256;

// 1024 * m / n orders the ratios m / n (m <= n <= 32) exactly: two distinct ones differ by at least 1 / (32 * 31),
// i.e. by more than one unit after the scaling, and equal ones give the same integer.  n = 0 has m = 0: ratio 0.
__device__ __forceinline__ uint32_t pck_rank(uint32_t m, uint32_t n) { return (m * 1024u) / (n ? n : 1u); }

struct GTTile {
    double x[kAPMaxGT][kAPMaxJoints];
    double y[kAPMaxGT][kAPMaxJoints];
    double head[kAPMaxGT];                  // head_scale * sqrt(hx * hx + hy * hy)
    uint32_t valid[kAPMaxGT];               // bit j: joint j annotated
    uint32_t n_valid[kAPMaxGT];
    unsigned long long best[kAPMaxGT];      // (rank << 32) | ~slot of the best prediction claiming this GT person
};

// One prediction (slot i) against every GT person: the warp's lane j evaluates joint j.  Returns the first GT person
// of maximal PCKh (assignGTmulti's row arg-max), its rank and the match mask against it.
__device__ __forceinline__ void best_gt(const GTTile& s, int G, bool has_pr, double xp, double yp, double thr, int lane,
                                        int* best_g, uint32_t* best_rank, uint32_t* best_mask) {
    int bg = 0;
    uint32_t br = 0, bm = 0;
    for (int g = 0; g < G; ++g) {
        bool hit = false;
        if (has_pr && ((s.valid[g] >> lane) & 1u)) {
            const double dx = __dsub_rn(xp, s.x[g][lane]), dy = __dsub_rn(yp, s.y[g][lane]);
            const double d = __ddiv_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))), s.head[g]);
            hit = d <= thr;                                  // NaN never matches
        }
        const uint32_t mask = __ballot_sync(0xffffffffu, hit);
        const uint32_t r = pck_rank(__popc(mask), s.n_valid[g]);
        if (g == 0 || r > br) { bg = g; br = r; bm = mask; }
    }
    *best_g = bg; *best_rank = br; *best_mask = bm;
}

__global__ void __launch_bounds__(kMatchThreads) ap_match_kernel(APMatchArgs a) {
    __shared__ GTTile s;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int J = a.J, Jp = min(a.K - 1, J);
    const int count = a.count[b];
    const int used = max(0, min(count, a.R));
    const int g0 = a.person_off[b], g1 = a.person_off[b + 1];
    const bool bad_gt = g0 < 0 || g1 < g0 || g1 > a.n_gt_rows || g1 - g0 > kAPMaxGT;
    const int G = bad_gt ? 0 : g1 - g0;
    if (tid == 0) {
        a.used[b] = used;
        a.flags[b] = (count > a.R ? APFLAG_OVERFLOW : 0) | (bad_gt ? APFLAG_BAD_GT : 0);
    }
    for (int g = tid; g < G; g += kMatchThreads) {
        const double* hb = a.head_box + 4 * (size_t)(g0 + g);
        const double hx = __dsub_rn(hb[2], hb[0]), hy = __dsub_rn(hb[3], hb[1]);
        s.head[g] = __dmul_rn(a.head_scale, __dsqrt_rn(__dadd_rn(__dmul_rn(hx, hx), __dmul_rn(hy, hy))));
        s.best[g] = 0ull;
        uint32_t v = 0;
        for (int j = 0; j < J; ++j) v |= (a.joint_valid[(size_t)(g0 + g) * J + j] != 0 ? 1u : 0u) << j;
        s.valid[g] = v;
        s.n_valid[g] = __popc(v);
    }
    for (int t = tid; t < G * J; t += kMatchThreads) {
        const int g = t / J, j = t - g * J;
        const double* p = a.joint_xy + 2 * ((size_t)(g0 + g) * J + j);
        s.x[g][j] = p[0];
        s.y[g][j] = p[1];
    }
    __syncthreads();
    if (tid < J) {                                           // annotated GT joints of the image (nGTall)
        int n = 0;
        for (int g = 0; g < G; ++g) n += (s.valid[g] >> tid) & 1u;
        a.n_gt[(size_t)b * J + tid] = n;
    }
    // A prediction's keypoint of joint j: the centre of part j + 1's box, (0, 0) where the part is absent
    // (evaluation.pred_frame); joints at or beyond K - 1 have no prediction at all.
    auto load_pred = [&](int i, bool* has_pr, double* xp, double* yp, float* score) {
        *has_pr = lane < Jp;
        float2 c = make_float2(0.0f, 0.0f);
        float sc = 0.0f;
        if (*has_pr) {
            const size_t e = ((size_t)b * a.R + i) * a.K + lane + 1;
            if (a.cell[e] >= 0) { c = box_centre(a.box[e]); sc = a.part_score[e]; }
        }
        *xp = (double)c.y; *yp = (double)c.x; *score = sc;
    };
    // pass 1: every prediction offers itself to its best GT person; each GT person keeps the first best offer
    if (G > 0) {
        for (int i = warp; i < used; i += kMatchThreads / 32) {
            bool has_pr; double xp, yp; float sc;
            load_pred(i, &has_pr, &xp, &yp, &sc);
            int bg; uint32_t br, bm;
            best_gt(s, G, has_pr, xp, yp, a.thresh, lane, &bg, &br, &bm);
            if (lane == 0 && br > 0) atomicMax(&s.best[bg], ((unsigned long long)br << 32) | (0xffffffffu - (uint32_t)i));
        }
    }
    __syncthreads();
    // pass 2: a prediction that won its best GT person is labelled with the match mask against it, any other with 0
    for (int i = warp; i < used; i += kMatchThreads / 32) {
        bool has_pr; double xp, yp; float sc;
        load_pred(i, &has_pr, &xp, &yp, &sc);
        uint32_t labels = 0;
        if (G > 0) {
            int bg; uint32_t br, bm;
            best_gt(s, G, has_pr, xp, yp, a.thresh, lane, &bg, &br, &bm);
            if (br > 0 && s.best[bg] == (((unsigned long long)br << 32) | (0xffffffffu - (uint32_t)i))) labels = bm;
        }
        if (has_pr) {
            const size_t o = ((size_t)b * a.R_out + i) * J + lane;
            a.score[o] = sc;
            a.label[o] = (uint8_t)((labels >> lane) & 1u);
        }
    }
}

// ---- finalize ----------------------------------------------------------------------------------------------------
// Entry offsets (exclusive scan of the used-slot counts, in image order), the joint segments of the key arrays, and
// the status counters; one CTA.
__global__ void __launch_bounds__(kScanThreads) ap_offsets_kernel(APFinalizeArgs a) {
    using Scan = cub::BlockScan<int, kScanThreads>;
    using Reduce = cub::BlockReduce<int, kScanThreads>;
    __shared__ typename Scan::TempStorage scan_tmp;
    __shared__ typename Reduce::TempStorage red_tmp;
    const int tid = threadIdx.x;
    int carry = 0, n_over = 0, n_bad = 0;
    for (int base = 0; base < a.N; base += kScanThreads) {
        const int b = base + tid;
        const int u = b < a.N ? a.used[b] : 0;
        if (b < a.N) {
            n_over += (a.flags[b] & APFLAG_OVERFLOW) != 0;
            n_bad += (a.flags[b] & APFLAG_BAD_GT) != 0;
        }
        int incl, tile_total;
        Scan(scan_tmp).InclusiveSum(u, incl, tile_total);
        if (b < a.N) a.offsets[b + 1] = carry + incl;
        carry += tile_total;
        __syncthreads();
    }
    n_over = Reduce(red_tmp).Sum(n_over);
    __syncthreads();
    n_bad = Reduce(red_tmp).Sum(n_bad);
    if (tid == 0) {
        a.offsets[0] = 0;
        a.status[0] = n_over;
        a.status[1] = n_bad;
        a.status[2] = carry;
    }
    for (int j = tid; j < a.Jp; j += kScanThreads) {
        a.seg_begin[j] = j * a.cap;
        a.seg_end[j] = j * a.cap + carry;
    }
}

// Score bits that order like the fp32 values, largest first when sorted descending: NaN above +inf (numpy sorts NaN
// last, so the reversed order puts it first), -0 equal to +0.
__device__ __forceinline__ unsigned long long score_bits(float v) {
    if (v != v) return 0xffffffffull;
    if (v == 0.0f) v = 0.0f;
    const uint32_t u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// One CTA per image: key = score bits | append ordinal | label.  The ordinal (the entry's position in image-then-slot
// order) is unique, so the keys are distinct and "descending key" is the pinned tie rule: equal scores, later entry
// first.
__global__ void __launch_bounds__(kKeyThreads) ap_keys_kernel(APFinalizeArgs a) {
    const int b = blockIdx.x;
    const int base = a.offsets[b], u = a.used[b];
    for (int t = threadIdx.x; t < u * a.Jp; t += kKeyThreads) {
        const int i = t / a.Jp, j = t - i * a.Jp;
        const size_t src = ((size_t)b * a.R + i) * a.J + j;
        const unsigned long long ord = (unsigned long long)(base + i);
        a.keys[(size_t)j * a.cap + base + i] = (score_bits(a.score[src]) << (a.ord_bits + 1)) | (ord << 1) | a.label[src];
    }
}

// computeRPC + VOCap of one joint over its sorted entries (descending key), one CTA per joint.  With npos_s the TPs at
// ranks <= s, prec_s = npos_s / (s + 1) and rec_s = npos_s / nGT, VOCap's sum over the recall steps is the sum over
// the TP ranks s of (rec_s - rec_{s-1}) * max(prec_s, ..., prec_{T-1}); the final step (1 - rec) multiplies a
// precision of 0.  The tiles are visited from the last rank to the first, so the running maximum of the precision
// and the count of later TPs are carried from tile to tile; every thread sums its terms in a fixed order and the
// block reduces them in a fixed order, so the result depends on the sorted entries alone.
__global__ void __launch_bounds__(kCurveThreads) ap_curve_kernel(APFinalizeArgs a, const unsigned long long* sorted) {
    using IntScan = cub::BlockScan<int, kCurveThreads>;
    using MaxScan = cub::BlockScan<double, kCurveThreads>;
    using IntReduce = cub::BlockReduce<long long, kCurveThreads>;
    using DblReduce = cub::BlockReduce<double, kCurveThreads>;
    __shared__ union {
        typename IntScan::TempStorage iscan;
        typename MaxScan::TempStorage mscan;
        typename IntReduce::TempStorage ired;
        typename DblReduce::TempStorage dred;
    } tmp;
    const int j = blockIdx.x, tid = threadIdx.x;
    const int T = j < a.Jp ? a.status[2] : 0;
    const unsigned long long* keys = sorted + (size_t)j * a.cap;

    long long ngt_part = 0;
    for (int b = tid; b < a.N; b += kCurveThreads) ngt_part += a.n_gt[(size_t)b * a.J + j];
    long long tp_part = 0;
    for (int s = tid; s < T; s += kCurveThreads) tp_part += (long long)(keys[s] & 1ull);
    const long long n_gt = IntReduce(tmp.ired).Sum(ngt_part);
    __syncthreads();
    const long long total_tp = IntReduce(tmp.ired).Sum(tp_part);
    __shared__ long long sh_ngt, sh_tp;
    if (tid == 0) { sh_ngt = n_gt; sh_tp = total_tp; }
    __syncthreads();
    const double ngt_d = (double)sh_ngt;
    const long long total = sh_tp;

    constexpr int kTile = kCurveThreads * kCurveItems;
    int tp_after = 0;                  // TPs at ranks beyond the current tile
    double run_max = 0.0;              // max precision beyond the current tile (VOCap's trailing 0 included)
    double sum = 0.0;
    for (int hi = T; hi > 0; hi -= kTile) {
        const int n = min(kTile, hi);
        int lab[kCurveItems], after[kCurveItems];
        double prec[kCurveItems], pmax[kCurveItems];
#pragma unroll
        for (int k = 0; k < kCurveItems; ++k) {
            const int q = tid * kCurveItems + k;              // q-th entry from the tile's end
            lab[k] = q < n ? (int)(keys[hi - 1 - q] & 1ull) : 0;
        }
        int tile_tp;
        IntScan(tmp.iscan).ExclusiveSum(lab, after, tile_tp);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kCurveItems; ++k) {
            const int q = tid * kCurveItems + k;
            const long long npos = total - (tp_after + after[k]);    // TPs at ranks <= s (the entry's own included)
            prec[k] = q < n ? __ddiv_rn((double)npos, (double)(hi - q)) : 0.0;
        }
        double tile_max;
        MaxScan(tmp.mscan).InclusiveScan(prec, pmax, cub::Max(), tile_max);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kCurveItems; ++k) {
            const int q = tid * kCurveItems + k;
            if (q < n && lab[k]) {
                const long long npos = total - (tp_after + after[k]);
                const double step = __dsub_rn(__ddiv_rn((double)npos, ngt_d), __ddiv_rn((double)(npos - 1), ngt_d));
                sum = __dadd_rn(sum, __dmul_rn(step, fmax(run_max, pmax[k])));
            }
        }
        tp_after += tile_tp;
        run_max = fmax(run_max, tile_max);
    }
    const double ap_sum = DblReduce(tmp.dred).Sum(sum);
    if (tid == 0) {
        if (T == 0) {                                        // no entries: computeMetrics' zeros
            a.ap[j] = 0.0; a.precision[j] = 0.0; a.recall[j] = 0.0;
        } else {
            const double nan = __longlong_as_double(0x7ff8000000000000ll);
            a.ap[j] = sh_ngt == 0 ? nan : __dmul_rn(ap_sum, 100.0);      // no GT joint: every recall is 0 / 0
            a.precision[j] = __dmul_rn(__ddiv_rn((double)total, (double)T), 100.0);
            a.recall[j] = __dmul_rn(__ddiv_rn((double)total, ngt_d), 100.0);
        }
    }
}

// the last entry of each result: the plain mean over the joints (a NaN joint makes it NaN)
__global__ void ap_mean_kernel(APFinalizeArgs a) {
    if (threadIdx.x < 3) {
        double* o = threadIdx.x == 0 ? a.ap : (threadIdx.x == 1 ? a.precision : a.recall);
        double s = 0.0;
        for (int j = 0; j < a.J; ++j) s = __dadd_rn(s, o[j]);
        o[a.J] = __ddiv_rn(s, (double)a.J);
    }
}

}  // namespace

cudaError_t launch_ap_match(const APMatchArgs& a, int B, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    ap_match_kernel<<<B, kMatchThreads, 0, st>>>(a);
    return cudaGetLastError();
}

size_t ap_workspace_layout(long long N, long long R, int J, APWorkspace* w) {
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t cap = (size_t)N * R;
    size_t o = 0;
    w->offsets = o;   o += up((size_t)(N + 1) * sizeof(int32_t));
    w->seg_begin = o; o += up((size_t)J * sizeof(int32_t));
    w->seg_end = o;   o += up((size_t)J * sizeof(int32_t));
    w->keys_a = o;    o += up((size_t)J * cap * sizeof(unsigned long long));
    w->keys_b = o;    o += up((size_t)J * cap * sizeof(unsigned long long));
    w->sort_temp = o; o += kAPSortTempBytes;
    w->total = o;
    return o;
}

cudaError_t launch_ap_finalize(APFinalizeArgs a, unsigned long long* keys_b, void* sort_temp, cudaStream_t st) {
    cudaError_t e;
    ap_offsets_kernel<<<1, kScanThreads, 0, st>>>(a);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    const unsigned long long* sorted = a.keys;
    if (a.Jp > 0) {
        ap_keys_kernel<<<a.N, kKeyThreads, 0, st>>>(a);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        cub::DoubleBuffer<unsigned long long> db(a.keys, keys_b);
        const int end_bit = 33 + a.ord_bits;
        size_t temp = 0;
        e = cub::DeviceSegmentedRadixSort::SortKeysDescending(nullptr, temp, db, a.Jp * a.cap, a.Jp, a.seg_begin,
                                                              a.seg_end, 0, end_bit, st);
        if (e != cudaSuccess) return e;
        if (temp > kAPSortTempBytes) return cudaErrorMemoryAllocation;
        e = cub::DeviceSegmentedRadixSort::SortKeysDescending(sort_temp, temp, db, a.Jp * a.cap, a.Jp, a.seg_begin,
                                                              a.seg_end, 0, end_bit, st);
        if (e != cudaSuccess) return e;
        sorted = db.Current();
    }
    ap_curve_kernel<<<a.J, kCurveThreads, 0, st>>>(a, sorted);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    ap_mean_kernel<<<1, 32, 0, st>>>(a);
    return cudaGetLastError();
}

}  // namespace ppn
