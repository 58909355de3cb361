// Device-side helpers shared by the PPN parser kernels (sm_100a).
//
// Exact arithmetic: every fp32 operation that the reference evaluates in numpy is written
// with the __f*_rn intrinsics, which round once and are never contracted into FMAs, so the
// results are bit-identical to numpy's regardless of compiler flags.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ppn {

// Track orders (config.py:67-80) carried by value in kernel arguments.
struct ChainTable {
    int32_t n_chains;
    int32_t parallel_ok;    // 1: every part has one limb and one predecessor, chains may be walked concurrently
    uint8_t off[33];        // PPN_MAX_CHAINS + 1
    uint8_t limb[192];      // PPN_MAX_CHAIN_STEPS
    uint8_t part[192];
};

struct Geom {               // per-launch constants derived from PPNShape
    int32_t B, K, E, H, W, HW, sH, sW, S, C;
    int32_t off_h, off_w;
    float gridW, gridH, inW, inH;
    size_t img_stride;      // C*HW floats
    size_t limb_off;        // 6*K*HW floats
    uint32_t magic_W, magic_K;   // ceil(2^32 / d) for exact x / d, 0 <= x < 65536 (0 when d == 1)
    int32_t dtype;               // HeadDtype of the head tensor (host side: picks the kernel instantiation)
    // optional device timeline (benchmarks: ppn_timeline): record `tl_slot` = {first CTA start, last CTA end,
    // first CTA past its dependency wait, first CTA past phase `tl_phase` of the kernel} in %globaltimer nanoseconds;
    // nullptr = off
    unsigned long long* tl;
    int32_t tl_slot;
    int32_t tl_phase;
};

enum : int { TL_START = 0, TL_END = 1, TL_WAITED = 2 };
__device__ __forceinline__ void tl_mark(const Geom& g, int what) {
    if (g.tl && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        unsigned long long* rec = g.tl + 4 * (size_t)g.tl_slot;
        if (what == TL_END) atomicMax(rec + 1, t); else atomicMin(rec + what, t);
    }
}

// phase boundaries inside a kernel, one per run (tune key "timeline.phase"): where a single image's latency goes
__device__ __forceinline__ void tl_phase(const Geom& g, int phase) {
    if (g.tl && threadIdx.x == 0 && g.tl_phase == phase) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (phase >= 100) atomicMax(g.tl + 4 * (size_t)g.tl_slot + 3, t);      // 100+: the LAST CTA past the point
        else atomicMin(g.tl + 4 * (size_t)g.tl_slot + 3, t);
    }
}

// the same from any warp (lane 0): phase boundaries of code that runs warp by warp
__device__ __forceinline__ void tl_phase_warp(const Geom& g, int phase) {
    if (g.tl && (threadIdx.x & 31) == 0 && g.tl_phase == phase) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        atomicMin(g.tl + 4 * (size_t)g.tl_slot + 3, t);
    }
}

// ---- head element types ------------------------------------------------------------------
// The head tensor may be fp32 (the reference's), fp16 or bf16 (a head emitted in 16 bits halves the
// HBM traffic of this path, SURVEY §8f row 1).  Every element is widened to fp32 — exactly — the
// moment it is loaded; all arithmetic after that is the fp32 arithmetic of the reference, so the
// result equals the reference run on `head.float()`.
enum HeadDtype : int { HEAD_F32 = 0, HEAD_F16 = 1, HEAD_BF16 = 2 };

__device__ __forceinline__ float widen(float v) { return v; }
__device__ __forceinline__ float widen(__half v) { return __half2float(v); }
__device__ __forceinline__ float widen(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T>
__device__ __forceinline__ float ldf(const T* p) { return widen(__ldg(p)); }      // read-only path + widen

// fp32 -> the element type, rounded once to nearest even; beyond the type's range +-inf (torch's .to())
template <typename T> __device__ __forceinline__ T narrow(float v) { return v; }
template <> __device__ __forceinline__ __half narrow<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 narrow<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
__device__ __forceinline__ uint32_t bits16(__half v) { return __half_as_ushort(v); }
__device__ __forceinline__ uint32_t bits16(__nv_bfloat16 v) { return __bfloat16_as_ushort(v); }
// two narrowed values as one 32-bit word, `lo` at the lower address
template <typename T> __device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    return bits16(narrow<T>(lo)) | (bits16(narrow<T>(hi)) << 16);
}

// torch.sigmoid's fp32 expression, 1 / (1 + exp(-x)): libdevice expf, one add, one IEEE division.  Shared by the
// fused head (model.py:133-136) and the loss on logits, so that a model trained through the one is parsed through
// the other with the same values; -inf gives 0, +inf gives 1.
__device__ __forceinline__ float sigmoid_f32(float x) { return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x))); }

// ---- the reference's cell arithmetic --------------------------------------------------
// delta = resp * conf  (rt_test.py:130)
template <typename T>
__device__ __forceinline__ float delta_at(const T* __restrict__ img, const Geom& g, int k, int c) {
    return __fmul_rn(ldf(img + (size_t)k * g.HW + c), ldf(img + (size_t)(g.K + k) * g.HW + c));
}

// (ymin, xmin, ymax, xmax) from the four raw head values of a cell at (row h, col w)
// (datatest.py:63-71, 80-85): two roundings for the centre (add, then multiply), one for the size,
// an exact halving, one for each corner.
__device__ __forceinline__ float4 box_from(float x, float y, float bw, float bh, int h, int w, const Geom& g) {
    const float rx = __fmul_rn(__fadd_rn(x, (float)w), g.gridW);
    const float ry = __fmul_rn(__fadd_rn(y, (float)h), g.gridH);
    const float hw = __fmul_rn(__fmul_rn(g.inW, bw), 0.5f);     // rw / 2 (exact halving)
    const float hh = __fmul_rn(__fmul_rn(g.inH, bh), 0.5f);
    return make_float4(__fsub_rn(ry, hh), __fsub_rn(rx, hw), __fadd_rn(ry, hh), __fadd_rn(rx, hw));
}

// the same for part k at cell c, reading the head tensor of one image
template <typename T>
__device__ __forceinline__ float4 box_at(const T* __restrict__ img, const Geom& g, int k, int c) {
    const int h = c / g.W, w = c - h * g.W;
    const size_t HW = g.HW;
    return box_from(ldf(img + (size_t)(2 * g.K + k) * HW + c), ldf(img + (size_t)(3 * g.K + k) * HW + c),
                    ldf(img + (size_t)(4 * g.K + k) * HW + c), ldf(img + (size_t)(5 * g.K + k) * HW + c), h, w, g);
}

// centre (y, x) of a (ymin, xmin, ymax, xmax) box, y = (ymin + ymax) / 2, x = (xmin + xmax) / 2 in fp32 (an add and
// an exact halving): the keypoint of a part (datatest.py:200-211, 314-317).  Shared by ppn_part_centres and the AP
// matcher (ppn_eval.cu), so that the evaluator scores exactly the points the evaluation frames carry.
__device__ __forceinline__ float2 box_centre(const float4 b) {
    return make_float2(__fmul_rn(__fadd_rn(b.x, b.z), 0.5f), __fmul_rn(__fadd_rn(b.y, b.w), 0.5f));
}

// numpy's maximum / minimum: propagate NaN (datatest.py:145-146)
__device__ __forceinline__ float np_max(float a, float b) { return (a >= b || a != a) ? a : b; }
__device__ __forceinline__ float np_min(float a, float b) { return (a <= b || a != a) ? a : b; }

// IoU >= thr of a tested box against an already kept one  (datatest.py:145-150).
// `thr_positive` (thr > 0, uniform) allows an exact shortcut: without overlap the reference's
// intersection is prod * 0, so its IoU is +-0 or NaN, and neither is >= a positive threshold —
// the division can be skipped without changing the answer.
__device__ __forceinline__ bool suppresses(const float4 tested, float area_tested,
                                           const float4 kept, float area_kept, float thr, bool thr_positive) {
    const float tly = np_max(tested.x, kept.x), tlx = np_max(tested.y, kept.y);
    const float bry = np_min(tested.z, kept.z), brx = np_min(tested.w, kept.w);
    const bool overlap = tly < bry && tlx < brx;
    if (thr_positive && !overlap) return false;
    const float prod = __fmul_rn(__fsub_rn(bry, tly), __fsub_rn(brx, tlx));
    const float inter = __fmul_rn(prod, overlap ? 1.0f : 0.0f);
    const float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_tested, area_kept), inter));
    return iou >= thr;      // NaN compares false: not suppressed
}

__device__ __forceinline__ float box_area(const float4 b) {
    return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));   // datatest.py:141
}

// ---- numpy argmax semantics -------------------------------------------------------------
// Sequential rule: a later element replaces the running best iff !(v <= best) and best is not
// NaN (first maximum wins; the first NaN wins and ends the scan).
__device__ __forceinline__ void argmax_step(float& best, int& idx, float v, int a) {
    const bool take = !(v <= best) && (best == best);
    best = take ? v : best;
    idx = take ? a : idx;
}

// Merge of two partial results over disjoint index sets: does (v2, i2) beat (v1, i1)?
__device__ __forceinline__ bool argmax_beats(float v2, int i2, float v1, int i1) {
    const bool n1 = v1 != v1, n2 = v2 != v2;
    if (n1 || n2) return n2 && (!n1 || i2 < i1);
    return v2 > v1 || (v2 == v1 && i2 < i1);
}

// ---- mbarrier / bulk-copy (TMA) PTX ----------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "PPN_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra PPN_DONE;\n"
        "bra PPN_WAIT;\n"
        "PPN_DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier; evict-first in
// L2 because the limb block is read exactly once.  bytes % 16 == 0, both addresses 16 B aligned.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    const uint64_t evict_first = 0x12F0000000000000ull;
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(evict_first) : "memory");
}
// Programmatic dependent launch (PDL): let the next kernel in the stream start its prologue /
// wait until every kernel this one depends on has completed and flushed.  Both are no-ops when
// the kernel was launched without a programmatic dependency.
enum : int {
    PDL_TRIGGER = 1,       // let the next kernel in the stream become resident now
    PDL_WAIT_START = 2,    // wait for the previous kernel before reading anything it (or a producer) wrote
    PDL_WAIT_END = 4,      // wait for the previous kernel before completing (keeps completion transitive)
};
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Ask the L2 to fetch a contiguous range (bytes % 16 == 0, 16 B aligned): later scattered reads of
// it then cost an L2 hit instead of a DRAM sector each.
__device__ __forceinline__ void bulk_prefetch_l2(const void* src_gmem, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int n_threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}
// streaming 128-bit load that does not allocate in L1
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

}  // namespace ppn
