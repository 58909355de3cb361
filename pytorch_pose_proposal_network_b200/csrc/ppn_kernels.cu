// The four kernels of the PPN output parser, hand-written for sm_100a (B200).
//
//   K3 limb_argmax_*      streams the limb block once and keeps the arg-max of every window
//                         (>= 92 % of all bytes; HBM-bound)           datatest.py:100,113
//   K1 decode_candidates  resp*conf, threshold, ordered compaction, box  datatest.py:63-92
//   K2 nms_*              greedy IoU suppression per box list           datatest.py:134-160
//   K4 tree_parse         walk the track orders from every kept root    datatest.py:103-131
//
// Launchers at the bottom are called by ppn_capi.cu.
#include <algorithm>
#include <atomic>
#include <mutex>

#include "ppn_kernels.h"

namespace ppn {

// =========================================================================================
// K3 — limb window arg-max
// =========================================================================================
// One (image, limb) "matrix" is S rows (window positions) by HW columns (cells), contiguous in
// the head tensor, and the answer is the column-wise arg-max.  Rows are contiguous, so any run
// of rows is one contiguous byte range: the producer thread moves such runs into a
// shared-memory ring with 1-D bulk copies (TMA engine, completion on an mbarrier), and the
// consumer threads reduce them from shared memory.  Thread (g, cv) owns float4 column cv and
// every G-th row of each chunk; the G partial results per column are merged once per matrix.
// Persistent: grid = SM count x ctas_per_sm.  Work is handed out DYNAMICALLY: the producer draws the
// next matrix from a global ticket counter and passes its index to the consumers through the ring
// (s_item[stage], published by the mbarrier's release/acquire).  A CTA that becomes resident late —
// e.g. because an NCCL kernel holds its SM — then simply takes fewer matrices instead of delaying its
// fixed share (measured: static dealing lost 35 % with a concurrent all_gather), and the last wave
// has no tail.  The last CTA to finish resets the counter for the next launch.

struct Partial { float v; int32_t i; };

// split-matrix ring kernels: work item -> first matrix and number of matrices (see ArgmaxPlan::n_big)
__host__ __device__ __forceinline__ int item_first(const ArgmaxPlan& p, int item) {
    return item < p.n_big ? item * p.G : p.n_big * p.G + (item - p.n_big) * p.small_m;
}
__host__ __device__ __forceinline__ int item_size(const ArgmaxPlan& p, int item) { return item < p.n_big ? p.G : p.small_m; }
__host__ __device__ __forceinline__ int item_count(const ArgmaxPlan& p, int n_mats) {
    const int rest = n_mats - p.n_big * p.G;
    return p.n_big + (rest + p.small_m - 1) / p.small_m;
}

__global__ void __launch_bounds__(1024, 1)
limb_argmax_tma_kernel(const float* __restrict__ head, uint16_t* __restrict__ amax, Geom g, ArgmaxPlan p, int pdl,
                       int* __restrict__ ticket, int32_t* __restrict__ zero2) {
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* ring = smem;
    Partial* part = reinterpret_cast<Partial*>(smem + (size_t)p.stages * p.stage_bytes);   // [2][G][HW]
    uint64_t* full = reinterpret_cast<uint64_t*>(part + (size_t)2 * p.G * g.HW);
    uint64_t* empty = full + p.stages;
    int* s_item = reinterpret_cast<int*>(empty + p.stages);                                // [stages]

    const int tid = threadIdx.x;
    const int n_cons = p.threads_padded;                 // consumer threads incl. idle lanes of the last warp
    const int n_mats = g.B * g.E;

    tl_mark(g, TL_START);
    if (tid == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], n_cons / 32);
        }
        fence_mbar_init();
    }
    if (pdl & PDL_WAIT_START) pdl_wait();                // default chain: `head` may come from the kernel before us
    if (zero2 && blockIdx.x == 0 && tid == 0) { zero2[0] = 0; zero2[1] = 0; }   // the parse kernel's dense-entry cursor
    if (pdl & PDL_TRIGGER) pdl_launch_dependents();      // the parse kernel may start its prologue now
    __syncthreads();

    if (tid >= n_cons) {
        // ---------------- producer: one thread feeds the ring ----------------
        if (tid == n_cons) {
            int stage = 0;
            uint32_t phase = 0;
            for (int m = ticket ? atomicAdd(ticket, 1) : (int)blockIdx.x;; m = ticket ? atomicAdd(ticket, 1) : m + (int)gridDim.x) {
                if (m >= n_mats) {                                   // no work left: tell the consumers
                    mbar_wait(&empty[stage], phase ^ 1u);
                    s_item[stage] = -1;
                    mbar_arrive(&full[stage]);
                    break;
                }
                const int b = m / g.E, ei = m - b * g.E;
                const float* src = head + (size_t)b * g.img_stride + g.limb_off + (size_t)ei * g.S * g.HW;
                for (int c = 0; c < p.chunks; ++c) {
                    mbar_wait(&empty[stage], phase ^ 1u);
                    if (c == 0) s_item[stage] = m;
                    const int rows = min(p.rows, g.S - c * p.rows);
                    const uint32_t bytes = (uint32_t)rows * g.HW * 4u;
                    mbar_arrive_expect_tx(&full[stage], bytes);
                    bulk_g2s(ring + (size_t)stage * p.stage_bytes, src + (size_t)c * p.rows * g.HW, bytes, &full[stage]);
                    if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                }
            }
            if (ticket && atomicAdd(ticket + 1, 1) == (int)gridDim.x - 1) { ticket[0] = 0; ticket[1] = 0; }
        }
        return;
    }

    // ---------------- consumers ----------------
    const bool active = tid < p.threads;
    const int grp = tid / p.CV, cv = tid - grp * p.CV;
    const int lane = tid & 31;
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0;; ++it) {
        mbar_wait(&full[stage], phase);
        const int m = s_item[stage];
        if (m < 0) break;
        float b0 = -INFINITY, b1 = -INFINITY, b2 = -INFINITY, b3 = -INFINITY;
        int i0 = 0, i1 = 0, i2 = 0, i3 = 0;
        for (int c = 0; c < p.chunks; ++c) {
            if (c > 0) mbar_wait(&full[stage], phase);
            if (active && !p.dry) {
                const int rows = min(p.rows, g.S - c * p.rows);
                const float4* col = reinterpret_cast<const float4*>(ring + (size_t)stage * p.stage_bytes) + cv;
                int a = c * p.rows + grp;
                int r = grp;
#pragma unroll 1
                for (; r + 3 * p.G < rows; r += 4 * p.G, a += 4 * p.G) {
                    const float4 v0 = col[(size_t)r * p.CV];
                    const float4 v1 = col[(size_t)(r + p.G) * p.CV];
                    const float4 v2 = col[(size_t)(r + 2 * p.G) * p.CV];
                    const float4 v3 = col[(size_t)(r + 3 * p.G) * p.CV];
                    argmax_step(b0, i0, v0.x, a); argmax_step(b1, i1, v0.y, a);
                    argmax_step(b2, i2, v0.z, a); argmax_step(b3, i3, v0.w, a);
                    argmax_step(b0, i0, v1.x, a + p.G); argmax_step(b1, i1, v1.y, a + p.G);
                    argmax_step(b2, i2, v1.z, a + p.G); argmax_step(b3, i3, v1.w, a + p.G);
                    argmax_step(b0, i0, v2.x, a + 2 * p.G); argmax_step(b1, i1, v2.y, a + 2 * p.G);
                    argmax_step(b2, i2, v2.z, a + 2 * p.G); argmax_step(b3, i3, v2.w, a + 2 * p.G);
                    argmax_step(b0, i0, v3.x, a + 3 * p.G); argmax_step(b1, i1, v3.y, a + 3 * p.G);
                    argmax_step(b2, i2, v3.z, a + 3 * p.G); argmax_step(b3, i3, v3.w, a + 3 * p.G);
                }
                for (; r < rows; r += p.G, a += p.G) {
                    const float4 v = col[(size_t)r * p.CV];
                    argmax_step(b0, i0, v.x, a); argmax_step(b1, i1, v.y, a);
                    argmax_step(b2, i2, v.z, a); argmax_step(b3, i3, v.w, a);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
        uint16_t* dst = amax + (size_t)m * g.HW;
        if (p.dry) continue;
        if (p.G == 1) {
            if (active) {
                const uint32_t lo = (uint32_t)i0 | ((uint32_t)i1 << 16), hi = (uint32_t)i2 | ((uint32_t)i3 << 16);
                *reinterpret_cast<uint2*>(dst + 4 * cv) = make_uint2(lo, hi);
            }
        } else {
            Partial* mine = part + (size_t)(it & 1) * p.G * g.HW;
            if (active) {
                Partial* row = mine + (size_t)grp * g.HW + 4 * cv;
                row[0] = Partial{b0, i0}; row[1] = Partial{b1, i1};
                row[2] = Partial{b2, i2}; row[3] = Partial{b3, i3};
            }
            named_bar_sync(1, n_cons);
            for (int c = tid; c < g.HW; c += n_cons) {
                Partial best = mine[c];
                for (int q = 1; q < p.G; ++q) {
                    const Partial o = mine[(size_t)q * g.HW + c];
                    if (argmax_beats(o.v, o.i, best.v, best.i)) best = o;
                }
                dst[c] = (uint16_t)best.i;
            }
            // `part` is double-buffered on the matrix parity, so one barrier per matrix is enough:
            // a thread can only overwrite buffer (it & 1) two matrices later, after the barrier of
            // matrix it+1, which every thread reaches only after finishing this merge.
        }
    }
    // In the PDL chain this kernel started without waiting for decode+NMS (it does not read their
    // output); it must not COMPLETE before they do, because the tree parse waits only for us.
    tl_mark(g, TL_END);
    if ((pdl & PDL_WAIT_END) && tid == 0) pdl_wait();
}

// Ring, second thread mapping, for SMALL matrices (S*HW*4 below ~64 KB): instead of splitting the
// rows of one matrix over G thread groups (which costs a merge and a barrier per matrix), the G
// groups take G different matrices.  Thread (j, cv) owns float4 column cv of matrix j of the
// current item for ALL rows, so there is nothing to merge and no barrier at all; each ring stage
// holds `rows` rows of each of the M = G matrices, brought in by M bulk copies issued by the
// lanes of the producer warp.
__global__ void __launch_bounds__(1024, 1)
limb_argmax_tma_multi_kernel(const float* __restrict__ head, uint16_t* __restrict__ amax, Geom g, ArgmaxPlan p, int pdl,
                             int* __restrict__ ticket, int32_t* __restrict__ zero2) {
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* ring = smem;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
    uint64_t* empty = full + p.stages;
    int* s_item = reinterpret_cast<int*>(empty + p.stages);                 // [stages] item index, -1 = no more work

    const int tid = threadIdx.x;
    const int n_cons = p.threads_padded;
    const int n_mats = g.B * g.E;
    const int n_items = item_count(p, n_mats);

    tl_mark(g, TL_START);
    if (tid == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], n_cons / 32);
        }
        fence_mbar_init();
    }
    if (pdl & PDL_WAIT_START) pdl_wait();                // default chain: `head` may come from the kernel before us
    if (zero2 && blockIdx.x == 0 && tid == 0) { zero2[0] = 0; zero2[1] = 0; }   // the parse kernel's dense-entry cursor
    if (pdl & PDL_TRIGGER) pdl_launch_dependents();      // the parse kernel may start its prologue now
    __syncthreads();

    if (tid >= n_cons) {
        // ---------------- producer warp: lane j fetches the rows of matrix j ----------------
        const int lane = tid - n_cons;
        int stage = 0;
        uint32_t phase = 0;
        int item = blockIdx.x;
        for (;;) {
            if (ticket) {                                            // lane 0 draws, the warp shares
                if (lane == 0) item = atomicAdd(ticket, 1);
                item = __shfl_sync(0xffffffffu, item, 0);
            }
            if (item >= n_items) {
                mbar_wait(&empty[stage], phase ^ 1u);
                if (lane == 0) { s_item[stage] = -1; mbar_arrive(&full[stage]); }
                break;
            }
            const int m0 = item_first(p, item);
            const int m = m0 + lane;
            const int nm = min(item_size(p, item), n_mats - m0);
            const int it_rows = item < p.n_big ? p.rows : p.rows_s, it_chunks = item < p.n_big ? p.chunks : p.chunks_s;
            const uint32_t it_slot = (uint32_t)it_rows * g.HW * 4u;
            const int b = m / g.E, ei = m - b * g.E;
            const float* src = head + (size_t)b * g.img_stride + g.limb_off + (size_t)ei * g.S * g.HW;
            for (int c = 0; c < it_chunks; ++c) {
                mbar_wait(&empty[stage], phase ^ 1u);
                const int rows = min(it_rows, g.S - c * it_rows);
                const uint32_t bytes = (uint32_t)rows * g.HW * 4u;
                if (lane == 0) {
                    if (c == 0) s_item[stage] = item;
                    mbar_arrive_expect_tx(&full[stage], bytes * nm);
                }
                __syncwarp();
                if (lane < nm)
                    bulk_g2s(ring + (size_t)stage * p.stage_bytes + (size_t)lane * it_slot,
                             src + (size_t)c * it_rows * g.HW, bytes, &full[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1u; }
            }
            if (!ticket) item += gridDim.x;
        }
        if (ticket && lane == 0 && atomicAdd(ticket + 1, 1) == (int)gridDim.x - 1) { ticket[0] = 0; ticket[1] = 0; }
        return;
    }

    // ---------------- consumers ----------------
    const int j = tid / p.CV, cv = tid - j * p.CV;
    const int lane = tid & 31;
    int stage = 0;
    uint32_t phase = 0;
    for (;;) {
        mbar_wait(&full[stage], phase);
        const int item = s_item[stage];
        if (item < 0) break;
        const int m = item_first(p, item) + j;
        const bool active = tid < p.threads && j < item_size(p, item) && m < n_mats;
        const int it_rows = item < p.n_big ? p.rows : p.rows_s, it_chunks = item < p.n_big ? p.chunks : p.chunks_s;
        const uint32_t it_slot = (uint32_t)it_rows * g.HW * 4u;
        float b0 = -INFINITY, b1 = -INFINITY, b2 = -INFINITY, b3 = -INFINITY;
        int i0 = 0, i1 = 0, i2 = 0, i3 = 0;
        for (int c = 0; c < it_chunks; ++c) {
            if (c > 0) mbar_wait(&full[stage], phase);
            if (active && !p.dry) {
                const int rows = min(it_rows, g.S - c * it_rows);
                const float4* col = reinterpret_cast<const float4*>(ring + (size_t)stage * p.stage_bytes + (size_t)j * it_slot) + cv;
                int a = c * it_rows;
                int r = 0;
#pragma unroll 1
                for (; r + 3 < rows; r += 4, a += 4) {
                    const float4 v0 = col[(size_t)r * p.CV];
                    const float4 v1 = col[(size_t)(r + 1) * p.CV];
                    const float4 v2 = col[(size_t)(r + 2) * p.CV];
                    const float4 v3 = col[(size_t)(r + 3) * p.CV];
                    argmax_step(b0, i0, v0.x, a); argmax_step(b1, i1, v0.y, a);
                    argmax_step(b2, i2, v0.z, a); argmax_step(b3, i3, v0.w, a);
                    argmax_step(b0, i0, v1.x, a + 1); argmax_step(b1, i1, v1.y, a + 1);
                    argmax_step(b2, i2, v1.z, a + 1); argmax_step(b3, i3, v1.w, a + 1);
                    argmax_step(b0, i0, v2.x, a + 2); argmax_step(b1, i1, v2.y, a + 2);
                    argmax_step(b2, i2, v2.z, a + 2); argmax_step(b3, i3, v2.w, a + 2);
                    argmax_step(b0, i0, v3.x, a + 3); argmax_step(b1, i1, v3.y, a + 3);
                    argmax_step(b2, i2, v3.z, a + 3); argmax_step(b3, i3, v3.w, a + 3);
                }
                for (; r < rows; ++r, ++a) {
                    const float4 v = col[(size_t)r * p.CV];
                    argmax_step(b0, i0, v.x, a); argmax_step(b1, i1, v.y, a);
                    argmax_step(b2, i2, v.z, a); argmax_step(b3, i3, v.w, a);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
        if (active && !p.dry) {
            const uint32_t lo = (uint32_t)i0 | ((uint32_t)i1 << 16), hi = (uint32_t)i2 | ((uint32_t)i3 << 16);
            *reinterpret_cast<uint2*>(amax + (size_t)m * g.HW + 4 * cv) = make_uint2(lo, hi);
        }
    }
    tl_mark(g, TL_END);
    if ((pdl & PDL_WAIT_END) && tid == 0) pdl_wait();    // see limb_argmax_tma_kernel
}

// The same ring and thread mapping for a 16-bit head (fp16 / bf16): rows are HW * 2 bytes and a
// thread owns EIGHT columns (one 16-byte vector).  Widening to fp32 is exact and monotone, so the
// values are compared in their packed 16-bit form, two columns per instruction: `v > best` as a
// per-half mask (HSET2), the running index (16 bits per column, S < 65536) updated through the mask
// (one LOP3), the running maximum by a NaN-propagating packed max (HMNMX2) — three instructions
// per two elements where the widened scalar form needed ten.  Signed zeros compare equal in both
// forms (first one wins).  NaN: numpy's arg-max returns the FIRST NaN of a column; here a NaN makes
// the running maximum NaN for good (and freezes the index), which is detected once per matrix and
// repaired by `first_nan16` — a plain scan of that column for its first NaN.  p.CV counts 16-byte
// vectors per row (HW / 8).
template <typename T16> struct Packed16;
template <> struct Packed16<__half> {
    using V2 = __half2;
    static constexpr uint32_t kNegInf2 = 0xFC00FC00u;
    static __device__ __forceinline__ bool is_nan(uint32_t h) { return (h & 0x7FFFu) > 0x7C00u; }
};
template <> struct Packed16<__nv_bfloat16> {
    using V2 = __nv_bfloat162;
    static constexpr uint32_t kNegInf2 = 0xFF80FF80u;
    static __device__ __forceinline__ bool is_nan(uint32_t h) { return (h & 0x7FFFu) > 0x7F80u; }
};

template <typename T16>
__device__ __forceinline__ void argmax_step2(uint32_t& best, uint32_t& idx, uint32_t v, uint32_t a2) {
    using V2 = typename Packed16<T16>::V2;
    const V2 bv = *reinterpret_cast<const V2*>(&best), vv = *reinterpret_cast<const V2*>(&v);
    const uint32_t m = __hgt2_mask(vv, bv);                 // 0xFFFF per half where v > best (false on NaN)
    idx = (idx & ~m) | (a2 & m);
    const V2 nb = __hmax2_nan(bv, vv);
    best = *reinterpret_cast<const uint32_t*>(&nb);
}

// index of the first NaN in column `col` of one S x HW matrix (the column is known to hold one)
template <typename T16>
__device__ __noinline__ int first_nan16(const T16* __restrict__ mat, int S, int HW, int col) {
    const uint16_t* p = reinterpret_cast<const uint16_t*>(mat) + col;
    for (int a = 0; a < S; ++a)
        if (Packed16<T16>::is_nan(__ldg(p + (size_t)a * HW))) return a;
    return 0;
}

template <typename T16>
__global__ void __launch_bounds__(1024, 1)
limb_argmax_tma_multi16_kernel(const T16* __restrict__ head, uint16_t* __restrict__ amax, Geom g, ArgmaxPlan p, int pdl,
                               int* __restrict__ ticket, int32_t* __restrict__ zero2) {
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* ring = smem;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
    uint64_t* empty = full + p.stages;
    int* s_item = reinterpret_cast<int*>(empty + p.stages);

    const int tid = threadIdx.x;
    const int n_cons = p.threads_padded;
    const int n_mats = g.B * g.E;
    const int n_items = item_count(p, n_mats);

    tl_mark(g, TL_START);
    if (tid == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], n_cons / 32);
        }
        fence_mbar_init();
    }
    if (pdl & PDL_WAIT_START) pdl_wait();
    if (zero2 && blockIdx.x == 0 && tid == 0) { zero2[0] = 0; zero2[1] = 0; }
    if (pdl & PDL_TRIGGER) pdl_launch_dependents();
    __syncthreads();

    if (tid >= n_cons) {
        const int lane = tid - n_cons;
        int stage = 0;
        uint32_t phase = 0;
        int item = blockIdx.x;
        for (;;) {
            if (ticket) {
                if (lane == 0) item = atomicAdd(ticket, 1);
                item = __shfl_sync(0xffffffffu, item, 0);
            }
            if (item >= n_items) {
                mbar_wait(&empty[stage], phase ^ 1u);
                if (lane == 0) { s_item[stage] = -1; mbar_arrive(&full[stage]); }
                break;
            }
            const int m0 = item_first(p, item);
            const int m = m0 + lane;
            const int nm = min(item_size(p, item), n_mats - m0);
            const int it_rows = item < p.n_big ? p.rows : p.rows_s, it_chunks = item < p.n_big ? p.chunks : p.chunks_s;
            const uint32_t it_slot = (uint32_t)it_rows * g.HW * 2u;
            const int b = m / g.E, ei = m - b * g.E;
            const T16* src = head + (size_t)b * g.img_stride + g.limb_off + (size_t)ei * g.S * g.HW;
            for (int c = 0; c < it_chunks; ++c) {
                mbar_wait(&empty[stage], phase ^ 1u);
                const int rows = min(it_rows, g.S - c * it_rows);
                const uint32_t bytes = (uint32_t)rows * g.HW * 2u;
                if (lane == 0) {
                    if (c == 0) s_item[stage] = item;
                    mbar_arrive_expect_tx(&full[stage], bytes * nm);
                }
                __syncwarp();
                if (lane < nm)
                    bulk_g2s(ring + (size_t)stage * p.stage_bytes + (size_t)lane * it_slot,
                             src + (size_t)c * it_rows * g.HW, bytes, &full[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1u; }
            }
            if (!ticket) item += gridDim.x;
        }
        if (ticket && lane == 0 && atomicAdd(ticket + 1, 1) == (int)gridDim.x - 1) { ticket[0] = 0; ticket[1] = 0; }
        return;
    }

    const int j = tid / p.CV, cv = tid - j * p.CV;
    const int lane = tid & 31;
    int stage = 0;
    uint32_t phase = 0;
    for (;;) {
        mbar_wait(&full[stage], phase);
        const int item = s_item[stage];
        if (item < 0) break;
        const int m = item_first(p, item) + j;
        const bool active = tid < p.threads && j < item_size(p, item) && m < n_mats;
        const int it_rows = item < p.n_big ? p.rows : p.rows_s, it_chunks = item < p.n_big ? p.chunks : p.chunks_s;
        const uint32_t it_slot = (uint32_t)it_rows * g.HW * 2u;
        uint32_t best[4], idx[4];                                   // two columns per register
#pragma unroll
        for (int q = 0; q < 4; ++q) { best[q] = Packed16<T16>::kNegInf2; idx[q] = 0u; }
        for (int c = 0; c < it_chunks; ++c) {
            if (c > 0) mbar_wait(&full[stage], phase);
            if (active && !p.dry) {
                const int rows = min(it_rows, g.S - c * it_rows);
                const uint4* col = reinterpret_cast<const uint4*>(ring + (size_t)stage * p.stage_bytes + (size_t)j * it_slot) + cv;
                uint32_t a2 = (uint32_t)(c * it_rows) * 0x00010001u;       // the row index in both halves
                int r = 0;
#pragma unroll 1
                for (; r + 3 < rows; r += 4, a2 += 0x00040004u) {
                    const uint4 r0 = col[(size_t)r * p.CV];
                    const uint4 r1 = col[(size_t)(r + 1) * p.CV];
                    const uint4 r2 = col[(size_t)(r + 2) * p.CV];
                    const uint4 r3 = col[(size_t)(r + 3) * p.CV];
                    argmax_step2<T16>(best[0], idx[0], r0.x, a2); argmax_step2<T16>(best[1], idx[1], r0.y, a2);
                    argmax_step2<T16>(best[2], idx[2], r0.z, a2); argmax_step2<T16>(best[3], idx[3], r0.w, a2);
                    argmax_step2<T16>(best[0], idx[0], r1.x, a2 + 0x00010001u); argmax_step2<T16>(best[1], idx[1], r1.y, a2 + 0x00010001u);
                    argmax_step2<T16>(best[2], idx[2], r1.z, a2 + 0x00010001u); argmax_step2<T16>(best[3], idx[3], r1.w, a2 + 0x00010001u);
                    argmax_step2<T16>(best[0], idx[0], r2.x, a2 + 0x00020002u); argmax_step2<T16>(best[1], idx[1], r2.y, a2 + 0x00020002u);
                    argmax_step2<T16>(best[2], idx[2], r2.z, a2 + 0x00020002u); argmax_step2<T16>(best[3], idx[3], r2.w, a2 + 0x00020002u);
                    argmax_step2<T16>(best[0], idx[0], r3.x, a2 + 0x00030003u); argmax_step2<T16>(best[1], idx[1], r3.y, a2 + 0x00030003u);
                    argmax_step2<T16>(best[2], idx[2], r3.z, a2 + 0x00030003u); argmax_step2<T16>(best[3], idx[3], r3.w, a2 + 0x00030003u);
                }
                for (; r < rows; ++r, a2 += 0x00010001u) {
                    const uint4 v = col[(size_t)r * p.CV];
                    argmax_step2<T16>(best[0], idx[0], v.x, a2); argmax_step2<T16>(best[1], idx[1], v.y, a2);
                    argmax_step2<T16>(best[2], idx[2], v.z, a2); argmax_step2<T16>(best[3], idx[3], v.w, a2);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
        if (active && !p.dry) {
            bool any_nan = false;
#pragma unroll
            for (int q = 0; q < 4; ++q)
                any_nan |= Packed16<T16>::is_nan(best[q] & 0xFFFFu) || Packed16<T16>::is_nan(best[q] >> 16);
            if (any_nan) {                                               // rare: repair the columns that hold a NaN
                const int b = m / g.E, ei = m - b * g.E;
                const T16* mat = head + (size_t)b * g.img_stride + g.limb_off + (size_t)ei * g.S * g.HW;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (Packed16<T16>::is_nan(best[q] & 0xFFFFu))
                        idx[q] = (idx[q] & 0xFFFF0000u) | (uint32_t)first_nan16<T16>(mat, g.S, g.HW, 8 * cv + 2 * q);
                    if (Packed16<T16>::is_nan(best[q] >> 16))
                        idx[q] = (idx[q] & 0x0000FFFFu) | ((uint32_t)first_nan16<T16>(mat, g.S, g.HW, 8 * cv + 2 * q + 1) << 16);
                }
            }
            *reinterpret_cast<uint4*>(amax + (size_t)m * g.HW + 8 * cv) = make_uint4(idx[0], idx[1], idx[2], idx[3]);
        }
    }
    tl_mark(g, TL_END);
    if ((pdl & PDL_WAIT_END) && tid == 0) pdl_wait();
}

// Variant without the ring: one CTA per matrix, 128-bit streaming loads straight to registers.
// Kept as the measured alternative (ppn_tune "argmax.variant" = 1).
__global__ void __launch_bounds__(1024, 1)
limb_argmax_ldg_kernel(const float* __restrict__ head, uint16_t* __restrict__ amax, Geom g, ArgmaxPlan p) {
    extern __shared__ __align__(128) unsigned char smem[];
    Partial* part = reinterpret_cast<Partial*>(smem);                  // [G][HW]
    const int tid = threadIdx.x;
    const int m = blockIdx.x;
    const int b = m / g.E, ei = m - b * g.E;
    const float4* src = reinterpret_cast<const float4*>(head + (size_t)b * g.img_stride + g.limb_off + (size_t)ei * g.S * g.HW);
    const bool active = tid < p.threads;
    const int grp = tid / p.CV, cv = tid - grp * p.CV;
    float b0 = -INFINITY, b1 = -INFINITY, b2 = -INFINITY, b3 = -INFINITY;
    int i0 = 0, i1 = 0, i2 = 0, i3 = 0;
    if (active) {
        const float4* col = src + cv;
        int r = grp;
        constexpr int U = 8;
#pragma unroll 1
        for (; r + (U - 1) * p.G < g.S; r += U * p.G) {
            float4 v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) v[u] = ldg_stream(col + (size_t)(r + u * p.G) * p.CV);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int a = r + u * p.G;
                argmax_step(b0, i0, v[u].x, a); argmax_step(b1, i1, v[u].y, a);
                argmax_step(b2, i2, v[u].z, a); argmax_step(b3, i3, v[u].w, a);
            }
        }
        for (; r < g.S; r += p.G) {
            const float4 v = ldg_stream(col + (size_t)r * p.CV);
            argmax_step(b0, i0, v.x, r); argmax_step(b1, i1, v.y, r);
            argmax_step(b2, i2, v.z, r); argmax_step(b3, i3, v.w, r);
        }
        Partial* row = part + (size_t)grp * g.HW + 4 * cv;
        row[0] = Partial{b0, i0}; row[1] = Partial{b1, i1};
        row[2] = Partial{b2, i2}; row[3] = Partial{b3, i3};
    }
    __syncthreads();
    uint16_t* dst = amax + (size_t)m * g.HW;
    for (int c = tid; c < g.HW; c += blockDim.x) {
        Partial best = part[c];
        for (int q = 1; q < p.G; ++q) {
            const Partial o = part[(size_t)q * g.HW + c];
            if (argmax_beats(o.v, o.i, best.v, best.i)) best = o;
        }
        dst[c] = (uint16_t)best.i;
    }
}

// Tiny batches (the reference's own deployment: one webcam frame at a time, rt_test.py:181-189): there
// are fewer matrices than SMs, so a matrix per CTA would leave most of the GPU idle and make the call's
// latency the time ONE SM needs to pull a whole matrix (1 MB at the native shape, ~20 us).  Here a
// thread-block CLUSTER of C CTAs shares one matrix: CTA r reduces rows [r*S/C, (r+1)*S/C) to a partial
// (max, index) per column in its shared memory, the cluster synchronises, and CTA 0 merges the C
// partials straight out of its peers' shared memory (distributed shared memory) — no workspace, no
// second launch.  Ties across CTAs go to the lower row, NaNs to the first one, like the in-CTA merge.
template <typename T> struct Vec4Of;
template <> struct Vec4Of<float> { using type = float4; };
template <> struct Vec4Of<__half> { using type = uint2; };
template <> struct Vec4Of<__nv_bfloat16> { using type = uint2; };
__device__ __forceinline__ void widen4(const float4 r, float* v, float) { v[0] = r.x; v[1] = r.y; v[2] = r.z; v[3] = r.w; }
__device__ __forceinline__ void widen4(const uint2 r, float* v, __half) {
    const __half2* h = reinterpret_cast<const __half2*>(&r);
    const float2 a = __half22float2(h[0]), b = __half22float2(h[1]);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ void widen4(const uint2 r, float* v, __nv_bfloat16) {
    v[0] = __uint_as_float(r.x << 16); v[1] = __uint_as_float(r.x & 0xffff0000u);
    v[2] = __uint_as_float(r.y << 16); v[3] = __uint_as_float(r.y & 0xffff0000u);
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_nctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of `p` (a shared-memory address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t dsmem_addr(const void* p, uint32_t rank) {
    uint32_t out;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(out) : "r"(smem_u32(p)), "r"(rank));
    return out;
}
__device__ __forceinline__ Partial ld_dsmem_partial(uint32_t addr) {
    Partial o;
    asm volatile("ld.shared::cluster.v2.b32 {%0, %1}, [%2];" : "=f"(o.v), "=r"(o.i) : "r"(addr) : "memory");
    return o;
}

template <typename T>
__global__ void __launch_bounds__(1024, 1)
limb_argmax_cluster_kernel(const T* __restrict__ head, uint16_t* __restrict__ amax, Geom g, int CV, int G, int pdl,
                           int32_t* __restrict__ zero2, int ring_rows) {
    extern __shared__ __align__(128) unsigned char smem[];
    Partial* part = reinterpret_cast<Partial*>(smem);                    // [G][HW]; row 0 ends up as the CTA's result
    constexpr int NS = 4;                                                // ring stages (ring_rows > 0)
    using V4 = typename Vec4Of<T>::type;
    const int tid = threadIdx.x;
    const uint32_t rank = cluster_ctarank(), C = cluster_nctarank();
    const int m = blockIdx.x / C;
    tl_mark(g, TL_START);
    tl_phase(g, 121);
    if (pdl & PDL_WAIT_START) pdl_wait();
    tl_mark(g, TL_WAITED);
    if (zero2 && blockIdx.x == 0 && tid == 0) { zero2[0] = 0; zero2[1] = 0; }
    if (pdl & PDL_TRIGGER) pdl_launch_dependents();
    const int b = m / g.E, ei = m - b * g.E;
    const V4* src = reinterpret_cast<const V4*>(head + (size_t)b * g.img_stride + g.limb_off + (size_t)ei * g.S * g.HW);
    const int r_lo = (int)((long long)g.S * rank / C), r_hi = (int)((long long)g.S * (rank + 1) / C);
    const bool active = tid < CV * G;
    const int grp = tid / CV, cv = tid - grp * CV;
    if (ring_rows > 0) {
        // The CTA's rows are one contiguous slab of the limb block: thread 0 streams it through a 4-stage ring of 1-D
        // bulk copies (everything the ring holds is in flight at once — with 128-bit loads a thread had 8 rows in
        // flight, two rounds and a tail of single loads per CTA, each a DRAM round trip: 4.4 - 7.7 us for 128 KB),
        // every thread then reads its columns out of shared memory.
        uint64_t* full = reinterpret_cast<uint64_t*>(smem + (((size_t)G * g.HW * sizeof(Partial) + 15) & ~(size_t)15));
        uint64_t* empty = full + NS;
        unsigned char* ring = smem + (((size_t)G * g.HW * sizeof(Partial) + 16 * sizeof(uint64_t) + 127) & ~(size_t)127);
        const uint32_t row_bytes = (uint32_t)g.HW * (uint32_t)sizeof(T), stage_bytes = (uint32_t)ring_rows * row_bytes;
        const int n_rows = r_hi - r_lo, n_chunks = (n_rows + ring_rows - 1) / ring_rows;
        const unsigned char* slab = reinterpret_cast<const unsigned char*>(src) + (size_t)r_lo * row_bytes;
        if (tid == 0) {
            for (int st = 0; st < NS; ++st) { mbar_init(&full[st], 1); mbar_init(&empty[st], (uint32_t)(CV * G)); }
            fence_mbar_init();
        }
        __syncthreads();
        auto issue = [&](int c) {
            const uint32_t bytes = (uint32_t)min(ring_rows, n_rows - c * ring_rows) * row_bytes;
            mbar_arrive_expect_tx(&full[c % NS], bytes);
            bulk_g2s(ring + (size_t)(c % NS) * stage_bytes, slab + (size_t)c * stage_bytes, bytes, &full[c % NS]);
        };
        if (tid == 0) for (int c = 0; c < NS && c < n_chunks; ++c) issue(c);
        float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        int idx[4] = {r_lo, r_lo, r_lo, r_lo};                           // an empty row range must never win a tie
        for (int c = 0; c < n_chunks; ++c) {
            const int st = c % NS, ph = (c / NS) & 1;
            if (active) {
                mbar_wait(&full[st], (uint32_t)ph);
                const int l0 = c * ring_rows, l1 = min(n_rows, l0 + ring_rows);
                int lr = l0 + (grp - l0 % G + G) % G;                    // this group's first row of the chunk
                const V4* rows = reinterpret_cast<const V4*>(ring + (size_t)st * stage_bytes);
                for (; lr < l1; lr += G) {
                    float v[4];
                    widen4(rows[(size_t)(lr - l0) * CV + cv], v, T());
#pragma unroll
                    for (int q = 0; q < 4; ++q) argmax_step(best[q], idx[q], v[q], r_lo + lr);
                }
                mbar_arrive(&empty[st]);
            }
            if (tid == 0 && c + NS < n_chunks) {                         // the stage is free once every reader has left it
                mbar_wait(&empty[st], (uint32_t)ph);
                issue(c + NS);
            }
        }
        if (active) {
            tl_phase(g, 22);
            tl_phase(g, 122);
            Partial* row = part + (size_t)grp * g.HW + 4 * cv;
#pragma unroll
            for (int q = 0; q < 4; ++q) row[q] = Partial{best[q], idx[q]};
        }
    } else if (active) {
        float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        int idx[4] = {r_lo, r_lo, r_lo, r_lo};                           // an empty row range must never win a tie
        constexpr int U = 8;                                             // 128 B per thread in flight: latency is all there is here
        int r = r_lo + grp;
#pragma unroll 1
        for (; r + (U - 1) * G < r_hi; r += U * G) {
            V4 raw[U];
#pragma unroll
            for (int u = 0; u < U; ++u) raw[u] = __ldg(src + (size_t)(r + u * G) * CV + cv);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                float v[4];
                widen4(raw[u], v, T());
#pragma unroll
                for (int q = 0; q < 4; ++q) argmax_step(best[q], idx[q], v[q], r + u * G);
            }
        }
        for (; r < r_hi; r += G) {
            float v[4];
            widen4(__ldg(src + (size_t)r * CV + cv), v, T());
#pragma unroll
            for (int q = 0; q < 4; ++q) argmax_step(best[q], idx[q], v[q], r);
        }
        tl_phase(g, 22);
        tl_phase(g, 122);
        Partial* row = part + (size_t)grp * g.HW + 4 * cv;
#pragma unroll
        for (int q = 0; q < 4; ++q) row[q] = Partial{best[q], idx[q]};
    }
    __syncthreads();
    for (int c = tid; c < g.HW; c += blockDim.x) {                       // the CTA's own result in part[0][c]
        Partial bestp = part[c];
        for (int q = 1; q < G; ++q) {
            const Partial o = part[(size_t)q * g.HW + c];
            if (argmax_beats(o.v, o.i, bestp.v, bestp.i)) bestp = o;
        }
        part[c] = bestp;
    }
    tl_phase(g, 23);
    cluster_sync_all();
    tl_phase(g, 24);
    if (rank == 0) {
        uint16_t* dst = amax + (size_t)m * g.HW;
        for (int c = tid; c < g.HW; c += blockDim.x) {
            Partial bestp = part[c];
            for (uint32_t q = 1; q < C; ++q) {
                const Partial o = ld_dsmem_partial(dsmem_addr(&part[c], q));
                if (argmax_beats(o.v, o.i, bestp.v, bestp.i)) bestp = o;
            }
            dst[c] = (uint16_t)bestp.i;
        }
    }
    tl_phase(g, 25);
    cluster_sync_all();                                                   // peers' shared memory stays alive until CTA 0 has read it
    tl_mark(g, TL_END);
    if ((pdl & PDL_WAIT_END) && tid == 0) pdl_wait();
}

// Any shape (H*W not a multiple of 4, huge grids): one thread per column, scalar loads.
template <typename T>
__global__ void __launch_bounds__(256)
limb_argmax_generic_kernel(const T* __restrict__ head, uint16_t* __restrict__ amax, Geom g) {
    const int m = blockIdx.x;                                             // matrices on grid.x: no 65 535 limit
    const int c = blockIdx.y * blockDim.x + threadIdx.x;
    if (c >= g.HW) return;
    const int b = m / g.E, ei = m - b * g.E;
    const T* col = head + (size_t)b * g.img_stride + g.limb_off + (size_t)ei * g.S * g.HW + c;
    float best = -INFINITY;
    int idx = 0;
    for (int a = 0; a < g.S; ++a) argmax_step(best, idx, ldf(col + (size_t)a * g.HW), a);
    amax[(size_t)m * g.HW + c] = (uint16_t)idx;
}

// =========================================================================================
// K1 — decode + ordered compaction of candidates, one CTA per (image, part)
// =========================================================================================
template <typename T>
__global__ void __launch_bounds__(256)
decode_candidates_kernel(const T* __restrict__ head, Geom g, int n_parts, float thr,
                         int32_t* __restrict__ cand_cell, float* __restrict__ cand_score,
                         float4* __restrict__ cand_box, int32_t* __restrict__ cand_count) {
    __shared__ int warp_tot[8];
    __shared__ int base_s;
    const int b = blockIdx.x, k = blockIdx.y;
    const T* img = head + (size_t)b * g.img_stride;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t list = ((size_t)b * n_parts + k) * g.HW;
    if (tid == 0) base_s = 0;
    __syncthreads();
    for (int c0 = 0; c0 < g.HW; c0 += blockDim.x) {
        const int c = c0 + tid;
        float d = 0.0f;
        bool hit = false;
        if (c < g.HW) {
            d = delta_at(img, g, k, c);
            hit = d > thr;                                   // strict, datatest.py:89
        }
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) warp_tot[warp] = __popc(bal);
        __syncthreads();
        int off = base_s, total = 0;
        for (int wi = 0; wi < (int)(blockDim.x >> 5); ++wi) {
            const int t = warp_tot[wi];
            if (wi < warp) off += t;
            total += t;
        }
        if (hit) {
            const int slot = off + __popc(bal & ((1u << lane) - 1u));
            cand_cell[list + slot] = c;
            cand_score[list + slot] = d;
            cand_box[list + slot] = box_at(img, g, k, c);
        }
        __syncthreads();
        if (tid == 0) base_s += total;
        __syncthreads();
    }
    if (tid == 0) cand_count[(size_t)b * n_parts + k] = base_s;
}

// restore_xy / restore_size as stand-alone operators (datatest.py:63-71) over n_planes [H,W] planes
__global__ void __launch_bounds__(256)
restore_xy_kernel(const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ rx,
                  float* __restrict__ ry, size_t n, int HW, int W, float gridW, float gridH) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = (int)(i % HW);
    const int h = c / W, w = c - h * W;
    rx[i] = __fmul_rn(__fadd_rn(x[i], (float)w), gridW);
    ry[i] = __fmul_rn(__fadd_rn(y[i], (float)h), gridH);
}

__global__ void __launch_bounds__(256)
restore_size_kernel(const float* __restrict__ w, const float* __restrict__ h, float* __restrict__ rw,
                    float* __restrict__ rh, size_t n, float inW, float inH) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    rw[i] = __fmul_rn(inW, w[i]);
    rh[i] = __fmul_rn(inH, h[i]);
}

// =========================================================================================
// K2 — greedy IoU NMS, one CTA per box list, everything in shared memory
// =========================================================================================
// 1. rank sort by (score desc, index desc) — keys are unique, so the rank is a permutation;
// 2. the boxes are visited 32 at a time.  Inside a block of 32 the serial dependency is resolved by one
//    warp from the block's 32x32 DIAGONAL suppression bits (built up front, in parallel, for all blocks);
// 3. only the boxes a block KEEPS are then tested against the later blocks (all warps, one warp per
//    (kept box, later block of 32), the word is a ballot) and OR-ed into the `removed` words.
// A box that is suppressed never suppresses anything (datatest.py:143-152), so its row of the n x n
// suppression matrix is never needed: with m survivors of n boxes this evaluates ~ m*n/2 + 16n pairs
// instead of n*n/2 (the first version built the whole upper triangle: 3-5x the work at the BASELINE
// shapes, 22 KB of shared memory for it at 576 boxes against 2.4 KB now).
__device__ __forceinline__ unsigned long long score_key(float s, int idx) {
    unsigned u = __float_as_uint(s);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);          // monotone map of fp32 order
    return ((unsigned long long)u << 32) | (unsigned)idx;
}

constexpr int kNmsBuckets = 128;
struct NmsSmem {
    float4* sbox;                 // [stride] boxes in visiting order
    unsigned long long* key;      // [stride] sort keys of the unsorted list
    float* sarea;                 // [stride]
    int32_t* sidx;                // [stride] index into the unsorted list
    int32_t* rank;                // [stride] rank accumulators of the split counting sort
    unsigned* diag;               // [stride] bit t of diag[i]: box i suppresses box 32*(i/32) + t (t > i % 32)
    unsigned* rem;                // [32] removed set, one word per block of 32 boxes
    int32_t* ctl;                 // [4] {kept mask of the current block, survivors so far, done, -}
    float4* kbox;                 // [32] the current block's survivors, compacted: boxes
    float* karea;                 // [32]   and areas
    int32_t* above;               // [kNmsBuckets] bucket sort: boxes in higher buckets
    int32_t* cursor;              // [kNmsBuckets] bucket sort: counts, then fill cursors
    unsigned* wmm;                // [64] per-warp {min, max} of the keys' upper words
};

__host__ __device__ inline size_t nms_bytes_per_list(int stride) {
    return (size_t)stride * (sizeof(float4) + sizeof(unsigned long long) + sizeof(float) + 2 * sizeof(int32_t) + sizeof(unsigned)) +
           32 * (sizeof(float4) + sizeof(float)) + (32 + 4) * sizeof(int32_t) + (2 * kNmsBuckets + 64) * sizeof(int32_t);
}

__device__ __forceinline__ NmsSmem nms_carve(unsigned char* base, int stride) {
    NmsSmem s;
    s.sbox = reinterpret_cast<float4*>(base);
    s.kbox = s.sbox + stride;
    s.key = reinterpret_cast<unsigned long long*>(s.kbox + 32);      // key, sarea, rank: 16 contiguous bytes per box, reused
    s.sarea = reinterpret_cast<float*>(s.key + stride);              //   as the survivor list of the wavefront NMS
    s.rank = reinterpret_cast<int32_t*>(s.sarea + stride);
    s.sidx = s.rank + stride;
    s.diag = reinterpret_cast<unsigned*>(s.sidx + stride);
    s.rem = s.diag + stride;
    s.ctl = reinterpret_cast<int32_t*>(s.rem + 32);
    s.karea = reinterpret_cast<float*>(s.ctl + 4);
    s.above = reinterpret_cast<int32_t*>(s.karea + 32);
    s.cursor = s.above + kNmsBuckets;
    s.wmm = reinterpret_cast<unsigned*>(s.cursor + kNmsBuckets);
    return s;
}

// Same answer as suppresses() when no coordinate is NaN: fmaxf/fminf differ from numpy's
// maximum/minimum only in NaN propagation and in the sign of a zero result, and a zero's sign
// cannot change `tl < br` nor the final `iou >= thr` (see DESIGN.md, "NMS exactness").
__device__ __forceinline__ bool suppresses_finite(const float4 tested, float area_tested,
                                                  const float4 kept, float area_kept, float thr, bool thr_positive) {
    const float tly = fmaxf(tested.x, kept.x), tlx = fmaxf(tested.y, kept.y);
    const float bry = fminf(tested.z, kept.z), brx = fminf(tested.w, kept.w);
    const bool overlap = tly < bry && tlx < brx;
    if (thr_positive && !overlap) return false;
    const float prod = __fmul_rn(__fsub_rn(bry, tly), __fsub_rn(brx, tlx));
    const float inter = __fmul_rn(prod, overlap ? 1.0f : 0.0f);
    const float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_tested, area_kept), inter));
    return iou >= thr;
}

// Branch-free pre-classification of one IoU test (boxes without NaN coordinates, 1e-6 <= thr <= 1e6).  The exact rule
// is RN(inter / den) >= thr with an IEEE division; here the quotient comes from the approximate divide (2 ulp for
// |den| within [2^-126, 2^126], CUDA math API) and only answers that are 2^-18 (relative) clear of the threshold
// count: `yes` when surely >= thr, `amb` raised when neither side is sure (or den is outside [1e-18, 1e18], NaN
// included) — the caller then evaluates suppresses_finite() for that pair.  No divergent branch, no division
// sequence: four to eight of these pipeline in a warp, where the exact test is ~250 dependent cycles behind a branch
// (one image at the native shape: 32 boxes against 10 survivors took 2.9 us on the wavefront's critical path).
__device__ __forceinline__ bool boxes_overlap(const float4 a, const float4 b) {      // tl < br on both axes (datatest.py:148)
    return fmaxf(a.x, b.x) < fminf(a.z, b.z) && fmaxf(a.y, b.y) < fminf(a.w, b.w);
}
__device__ __forceinline__ bool iou_sure(const float4 tested, float area_tested, const float4 kept, float area_kept,
                                         float thr_lo, float thr_hi, bool& amb) {
    const float tly = fmaxf(tested.x, kept.x), tlx = fmaxf(tested.y, kept.y);
    const float bry = fminf(tested.z, kept.z), brx = fminf(tested.w, kept.w);
    const bool overlap = tly < bry && tlx < brx;
    const float prod = __fmul_rn(__fsub_rn(bry, tly), __fsub_rn(brx, tlx));
    const float inter = overlap ? prod : 0.0f;
    const float den = __fsub_rn(__fadd_rn(area_tested, area_kept), inter);
    const float q = __fdividef(inter, den);
    const bool in_range = fabsf(den) > 1e-18f && fabsf(den) < 1e18f;
    const bool yes = q > thr_hi, no = q < thr_lo;
    amb |= !(in_range && (yes || no));
    return yes;
}

constexpr int kNmsWalkMax = 12;      // resolve a block survivor by survivor when at most this many of its boxes are still alive
constexpr int NMS_BLOCKWISE = 128;   // launch bit of the decode+NMS and fused parse kernels: phase 3 block by block (see nms_core)

// Whole CTA.  Precondition: s.key[0..n) holds the keys of the n unsorted boxes `ubox` (global or
// shared), s.rank[0..n) is zero, and a __syncthreads() has made both visible.  Writes
// out[pos] = map ? map[idx] : idx for the kept boxes in visiting order and returns their number (in
// every thread).  n <= 1024.
__device__ __forceinline__ unsigned ld_acquire_cta_shared(const void* p) {
    unsigned v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"((unsigned)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_cta_shared(void* p, unsigned v) {
    asm volatile("st.release.cta.shared.u32 [%0], %1;" :: "r"((unsigned)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}

// `blockwise` (tune key "nms.blockwise", off by default): round 1/2's barrier-per-block phase 3 instead of the
// warp wavefront below — kept for A/B measurements and as a second implementation the tests compare.
__device__ __forceinline__ int nms_core(const NmsSmem& s, const float4* ubox, int n, float thr, int limit,
                                        int32_t* __restrict__ out, const int32_t* map, const Geom* tg = nullptr,
                                        bool blockwise = false, bool quick = true) {
    const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, n_warps = T >> 5;
    const int Wd = (n + 31) >> 5;
    // ---- 1. rank: every box's rank = number of larger keys ----------------------------------------------------
    if (!blockwise && n > 128) {                                    // (short lists: the four barriers cost more than the n x n count)
        // Bucket sort on the keys' upper words (the monotone image of the score): 128 buckets over [min, max] by a
        // shift, a histogram, one warp's suffix sums (= how many boxes lie in higher buckets), the keys regrouped by
        // bucket, and a box is only compared with the members of its OWN bucket.  Exact for any input — a skewed
        // distribution just makes buckets long (all scores equal: the old n x n count).  The n x n count was a quarter
        // of the decode+NMS kernel's instructions at 256 boxes per list and 4.5 us of one image's latency at 576.
        unsigned long long* tmp = reinterpret_cast<unsigned long long*>(s.sbox);      // written by the sort below, free until then
        unsigned lo = 0xffffffffu, hi = 0u;
        for (int i = tid; i < n; i += T) {
            const unsigned h = (unsigned)(s.key[i] >> 32);
            lo = min(lo, h);
            hi = max(hi, h);
        }
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        if (lane == 0) { s.wmm[2 * warp] = lo; s.wmm[2 * warp + 1] = hi; }
        for (int bk = tid; bk < kNmsBuckets; bk += T) s.cursor[bk] = 0;
        __syncthreads();
        for (int wv = 0; wv < n_warps; ++wv) { lo = min(lo, s.wmm[2 * wv]); hi = max(hi, s.wmm[2 * wv + 1]); }
        const int shift = max(0, 25 - __clz((int)(hi - lo)));      // (h - lo) >> shift < 128
        for (int i = tid; i < n; i += T) atomicAdd(&s.cursor[(((unsigned)(s.key[i] >> 32)) - lo) >> shift], 1);
        __syncthreads();
        if (warp == 0) {                                            // suffix sums over the buckets, 4 per lane
            int c[4], sum = 0;
#pragma unroll
            for (int u = 0; u < 4; ++u) { c[u] = s.cursor[4 * lane + u]; sum += c[u]; }
            int incl = sum;                                         // inclusive scan from the TOP lane down
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_down_sync(0xffffffffu, incl, o);
                if (lane + o < 32) incl += up;
            }
            int run = incl - sum;                                   // boxes in the buckets of higher lanes
#pragma unroll
            for (int u = 3; u >= 0; --u) {
                s.above[4 * lane + u] = run;
                s.cursor[4 * lane + u] = run;
                run += c[u];
            }
        }
        __syncthreads();
        for (int i = tid; i < n; i += T) {
            const unsigned long long k = s.key[i];
            tmp[atomicAdd(&s.cursor[(((unsigned)(k >> 32)) - lo) >> shift], 1)] = k;
        }
        __syncthreads();
        for (int i = tid; i < n; i += T) {
            const unsigned long long mine = s.key[i];
            const int bkt = (int)((((unsigned)(mine >> 32)) - lo) >> shift);
            const int p0 = s.above[bkt], p1 = s.cursor[bkt];        // the bucket's members (cursor ended at its end)
            int r = p0;
            for (int p2 = p0; p2 < p1; ++p2) r += (tmp[p2] > mine);
            s.rank[i] = r;
        }
    } else {
    int split = T / n;
    split = split < 1 ? 1 : (split > 8 ? 8 : split);
    const int chunk = (n + split - 1) / split;
    for (int item = tid; item < n * split; item += T) {
        const int part = item / n, i = item - part * n;
        const unsigned long long mine = s.key[i];
        const int j1 = min(n, (part + 1) * chunk);
        int r = 0;
        for (int j = part * chunk; j < j1; ++j) r += (s.key[j] > mine);
        if (split == 1) s.rank[i] = r; else atomicAdd(&s.rank[i], r);
    }
    }
    __syncthreads();
    if (tg) tl_phase(*tg, 11);
    bool has_nan = false;
    for (int i = tid; i < n; i += T) {
        const float4 bx = ubox[i];
        const int r = s.rank[i];
        has_nan |= (bx.x != bx.x) | (bx.y != bx.y) | (bx.z != bx.z) | (bx.w != bx.w);
        s.sbox[r] = bx;
        s.sarea[r] = box_area(bx);
        s.sidx[r] = i;
    }
    if (tid < 32) s.rem[tid] = 0u;
    if (tid == 0) s.ctl[0] = 0;
    const bool any_nan = __syncthreads_or(has_nan);
    const bool thr_pos = thr > 0.0f;
    if (tg) tl_phase(*tg, 12);
    // (tried, round 2: the FULL n x n suppression bit matrix built by all warps first, then either every box deciding
    //  for itself from its column, round after round, or one warp walking the survivors with ballot / find-first-set and
    //  OR-ing their rows into the removed set.  Exact both ways (the property tests keep a host model of the
    //  second), and slower both ways: all n^2/2 pair tests instead of survivors x rest, ~2 barrier rounds resp. ~210
    //  dependent cycles per SURVIVOR.  One image at the reference's native shape, 351 candidates -> 58 survivors:
    //  28 us block by block, 35 us with the matrix; 1024 dense images (256 -> 225): 91 -> 105 us.)
    // ---- 2. diagonal blocks: one warp per box i, lanes = the boxes of i's own block of 32 -----------------
    // `quick`: latency over instruction count.  iou_sure() costs ~28 instructions a pair where the exact test leaves
    // after ~10 when the boxes do not overlap at all: right for the one-CTA-per-image kernels, whose dependent chains
    // are what a small batch waits for, wrong for the throughput-bound decode+NMS grid of a dense crowd (1024 images of
    // 225 people: 72 -> 104 us with it).
    const bool fast_ok = quick && !any_nan && thr >= 1e-6f && thr <= 1e6f;
    const float thr_lo = thr * (1.0f - 3.8147e-6f), thr_hi = thr * (1.0f + 3.8147e-6f);
    if (fast_ok) {
        // two boxes i per warp and turn: independent, branch-free tests in flight together
        for (int i = warp; i < n; i += 2 * n_warps) {
            unsigned word[2], ambw = 0u;
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int ii = min(i + u * n_warps, n - 1);
                const int j = (ii & ~31) + lane, jj = min(j, n - 1);
                bool amb = false;
                const bool yes = iou_sure(s.sbox[jj], s.sarea[jj], s.sbox[ii], s.sarea[ii], thr_lo, thr_hi, amb);
                const bool valid = j > ii && j < n;
                word[u] = __ballot_sync(0xffffffffu, yes && valid);
                ambw |= __ballot_sync(0xffffffffu, amb && valid);
            }
            if (ambw) {                                               // rare: a quotient within 2^-18 of the threshold
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int ii = min(i + u * n_warps, n - 1);
                    const int j = (ii & ~31) + lane;
                    bool bit = false;
                    if (j > ii && j < n) bit = suppresses_finite(s.sbox[j], s.sarea[j], s.sbox[ii], s.sarea[ii], thr, thr_pos);
                    word[u] = __ballot_sync(0xffffffffu, bit);
                }
            }
#pragma unroll
            for (int u = 0; u < 2; ++u)
                if (lane == 0 && i + u * n_warps < n) s.diag[i + u * n_warps] = word[u];
        }
    } else {
        for (int i = warp; i < n; i += n_warps) {
            const float4 bi = s.sbox[i];
            const float ai = s.sarea[i];
            const int j = (i & ~31) + lane;
            bool bit = false;
            if (j > i && j < n) {
                const float4 bj = s.sbox[j];
                bit = any_nan ? suppresses(bj, s.sarea[j], bi, ai, thr, thr_pos)
                              : suppresses_finite(bj, s.sarea[j], bi, ai, thr, thr_pos);
            }
            const unsigned word = __ballot_sync(0xffffffffu, bit);
            if (lane == 0) s.diag[i] = word;
        }
    }
    __syncthreads();
    if (tg) tl_phase(*tg, 13);
    if (!blockwise) {
        // ---- 3. WAVEFRONT: a warp owns a word of 32 boxes (box = lane) from here to its verdict; no CTA barrier.
        //      The survivors so far are a list in shared memory that only grows, published together with the number
        //      of resolved words in ONE word (release / acquire).  A warp keeps testing its boxes against whatever
        //      survivors have been published — the earlier words' survivors, long before its predecessor is
        //      resolved — and when the count of resolved words reaches its own, it has seen every earlier survivor:
        //      it resolves its own 32-box dependency, appends its survivors and publishes.  On the critical path per
        //      word: notice the predecessor's survivors (a handful), test them, resolve, publish — the block-by-block
        //      version below pays two CTA barriers, a compaction by warp 0 and the whole cross phase per word.
        //      The resolve is not the 32-step chain either: the word's diagonal bits are transposed beforehand (5
        //      shuffle butterflies, off the critical path) so that lane t holds the EARLIER boxes that would suppress
        //      box t; then rounds of two ballots — a box with a kept suppressor dies, a box none of whose
        //      suppressors is still undecided is kept — as many rounds as the longest suppression chain (2-4).
        //      Survivors' boxes live in the 16 bytes per box of {sort keys, areas, ranks}, all dead by now; areas are
        //      recomputed (same operations, same bits).
        float4* kall = reinterpret_cast<float4*>(s.key);
        for (int w = warp; w < Wd; w += n_warps) {
            const int i0 = w << 5, nb = min(32, n - i0);
            const bool inb = lane < nb;
            const float4 bj = s.sbox[inb ? i0 + lane : i0];
            const float aj = box_area(bj);
            unsigned col = inb ? s.diag[i0 + lane] : 0u;               // row form: the later boxes of the word that box `lane` suppresses
#pragma unroll
            for (int sh = 16; sh >= 1; sh >>= 1) {                     // 32 x 32 bit transpose across the lanes
                const unsigned m = sh == 16 ? 0x0000ffffu : sh == 8 ? 0x00ff00ffu : sh == 4 ? 0x0f0f0f0fu : sh == 2 ? 0x33333333u : 0x55555555u;
                const unsigned other = __shfl_xor_sync(0xffffffffu, col, sh);
                col = (lane & sh) ? ((col & ~m) | ((other >> sh) & m)) : ((col & m) | ((other & m) << sh));
            }                                                          // column form: the earlier boxes of the word that suppress box `lane`
            bool dead = !inb;
            int seen = 0;
            bool fin = false;
            for (;;) {
                unsigned st = 0u;
                if (lane == 0) st = ld_acquire_cta_shared(&s.ctl[0]);
                st = __shfl_sync(0xffffffffu, st, 0);
                __syncwarp();
                const int m_pub = (int)(st & 0xffffu), wd = (int)((st >> 16) & 0x7fffu);
                fin = (st >> 31) != 0u;
                if (fin) break;
                if (m_pub > seen) {
                    bool exact = !fast_ok;
                    if (fast_ok && __any_sync(0xffffffffu, !dead)) {
                        bool hit = false, amb = false;                 // every lane, dead or not: nothing diverges
#pragma unroll 4
                        for (int q = seen; q < m_pub; ++q) {
                            const float4 kb = kall[q];
                            hit |= iou_sure(bj, aj, kb, box_area(kb), thr_lo, thr_hi, amb);
                        }
                        exact = __any_sync(0xffffffffu, amb && !hit && !dead);   // rare
                        if (!exact) dead |= hit;
                    }
                    if (exact && !dead) {
                        bool hit = false;
                        if (any_nan) {
                            for (int q = seen; q < m_pub; ++q) {
                                const float4 kb = kall[q];
                                hit |= suppresses(bj, aj, kb, box_area(kb), thr, thr_pos);
                            }
                        } else {
                            for (int q = seen; q < m_pub; ++q) {
                                const float4 kb = kall[q];
                                hit |= suppresses_finite(bj, aj, kb, box_area(kb), thr, thr_pos);
                            }
                        }
                        dead = hit;
                    }
                    seen = m_pub;
                }
                if (wd >= w) break;                                    // every earlier word is resolved, and `seen` covers their survivors
            }
            if (fin) break;
            if (tg) { if (w == 0) tl_phase_warp(*tg, 14); else if (w == 1) tl_phase_warp(*tg, 16); }
            unsigned und = ~__ballot_sync(0xffffffffu, dead);          // still to decide (lanes past the list count as dead)
            unsigned kept = 0u;
            while (und) {
                const bool mine = (und >> lane) & 1u;
                const bool killed = mine && (col & kept) != 0u;
                const bool free_ = mine && !killed && (col & und) == 0u;
                const unsigned k = __ballot_sync(0xffffffffu, free_);
                const unsigned d = __ballot_sync(0xffffffffu, killed);
                kept |= k;
                und &= ~(k | d);
            }
            bool done = false;
            if (limit > 0 && seen + __popc(kept) >= limit) {           // datatest.py:154-155
                int need = limit - seen;
                unsigned trimmed = 0u;
                for (unsigned rest = kept; need > 0 && rest; --need) { const unsigned low = rest & (0u - rest); trimmed |= low; rest ^= low; }
                kept = trimmed;
                done = true;
            }
            if ((kept >> lane) & 1u) {
                const int idx = s.sidx[i0 + lane];
                const int pos = seen + __popc(kept & ((1u << lane) - 1u));
                out[pos] = map ? map[idx] : idx;
                kall[pos] = bj;
            }
            __syncwarp();
            if (lane == 0)
                st_release_cta_shared(&s.ctl[0], ((done || w == Wd - 1) ? 0x80000000u : 0u) | ((unsigned)(w + 1) << 16) |
                                                     (unsigned)(seen + __popc(kept)));
            if (tg) {
                if (w == 0) tl_phase_warp(*tg, 15); else if (w == 1) tl_phase_warp(*tg, 17); else if (w == 2) tl_phase_warp(*tg, 18);
                if (w == Wd - 1) tl_phase_warp(*tg, 19);
            }
            if (done) break;
        }
        __syncthreads();
        return s.ctl[0] & 0xffff;
    }
    // ---- 3. block by block: warp 0 resolves the block, everybody tests its survivors against the rest ------
    int m = 0;
    for (int w = 0; w < Wd; ++w) {
        const int i0 = w << 5;
        if (warp == 0) {
            unsigned cur = s.rem[w];
            const int nb = min(32, n - i0);
            const unsigned valid = nb == 32 ? 0xffffffffu : ((1u << nb) - 1u);
            // (tried: the 32-step chain in ONE lane on words it loads itself instead of a shuffle per step — slower,
            //  decode+NMS 90.8 -> 103.4 us at the dense-crowd shape: the kernel has 40 registers and the words spill)
            const unsigned diag = (lane < nb) ? s.diag[i0 + lane] : 0u;
            unsigned kept = 0;
            unsigned open = ~cur & valid;                          // boxes of the block the earlier blocks left alive
            if (__popc(open) <= kNmsWalkMax) {
                // few of them (every block but the first ones when boxes overlap a lot): hop from survivor to survivor
                // with find-first-set, one dependent shuffle per SURVIVOR instead of one per box
                while (open) {
                    const int t = __ffs((int)open) - 1;
                    kept |= 1u << t;
                    open &= ~(__shfl_sync(0xffffffffu, diag, t) | (1u << t));
                }
            } else {
#pragma unroll
                for (int t = 0; t < 32; ++t) {
                    const unsigned d = __shfl_sync(0xffffffffu, diag, t);
                    const unsigned take = (~cur >> t) & 1u;
                    kept |= take << t;
                    cur |= d & (0u - take);
                }
                kept &= valid;
            }
            bool done = false;
            if (limit > 0 && m + __popc(kept) >= limit) {      // datatest.py:154-155
                int need = limit - m;
                unsigned trimmed = 0;
                for (unsigned rest = kept; need > 0 && rest; --need) { const unsigned low = rest & (0u - rest); trimmed |= low; rest ^= low; }
                kept = trimmed;
                done = true;
            }
            if ((kept >> lane) & 1u) {
                const int idx = s.sidx[i0 + lane];
                const int pos = __popc(kept & ((1u << lane) - 1u));
                out[m + pos] = map ? map[idx] : idx;
                s.kbox[pos] = s.sbox[i0 + lane];                  // the block's survivors, compacted for the phase below
                s.karea[pos] = s.sarea[i0 + lane];
            }
            if (lane == 0) { s.ctl[0] = (int)kept; s.ctl[1] = m + __popc(kept); s.ctl[2] = done || w == Wd - 1; }
        }
        __syncthreads();
        const unsigned kept = (unsigned)s.ctl[0];
        m = s.ctl[1];
        if (s.ctl[2]) break;                                      // uniform: limit reached or last block
        const int n_kept = __popc(kept);
        // A warp takes a whole WORD of later boxes, one box per lane, and runs over the block's survivors (compacted by
        // warp 0 above: broadcast reads of consecutive addresses, nothing in the loop depends on the previous turn but
        // the OR); one ballot and one plain store per word — a word has one writer per phase, so no atomics.
        // (Until round 2 it was the other way round — lanes held the survivors, the warps strode over the later boxes,
        // one vote and one shared-memory atomicOr per suppressed box: 32 x words turns instead of survivors x words, and
        // with a handful of survivors removing nearly everything behind them, 16 warps' atomics queueing on one or two
        // words.  1024 dense images, decode+NMS alone: 90.8 -> 77.4 us, the whole step 304 -> 270 us; one image of 351 candidates at the
        // native shape: 32.9 -> 31.6 us, where 16 warps' dependent instruction chains and 22 barriers are what is left.)
        if (n_kept == 0) { __syncthreads(); continue; }
        // When fewer words are left than there are warps, the survivors are split as well: G warps per word, each with
        // its share of them, OR-ed together with at most G atomics per word.
        const int n_words = Wd - w - 1;
        int G = n_words > 0 ? n_warps / n_words : 1;
        G = G < 1 ? 1 : (G > n_kept ? n_kept : G);
        const int chunk = (n_kept + G - 1) / G;
        for (int item = warp; item < n_words * G; item += n_warps) {
            const int grp = item / n_words, w2 = w + 1 + (item - grp * n_words);
            const int q0 = grp * chunk, q1 = min(n_kept, q0 + chunk);
            const int j = (w2 << 5) + lane;
            const unsigned remw = s.rem[w2];
            bool bit = false;
            if (j < n && !((remw >> lane) & 1u)) {
                const float4 bj = s.sbox[j];
                const float aj = s.sarea[j];
                if (any_nan) {
                    for (int q = q0; q < q1; ++q) bit |= suppresses(bj, aj, s.kbox[q], s.karea[q], thr, thr_pos);
                } else {
#pragma unroll 4
                    for (int q = q0; q < q1; ++q) bit |= suppresses_finite(bj, aj, s.kbox[q], s.karea[q], thr, thr_pos);
                }
            }
            const unsigned word = __ballot_sync(0xffffffffu, bit);
            if (lane == 0 && word) {
                if (G == 1) s.rem[w2] = remw | word; else atomicOr(&s.rem[w2], word);
            }
        }
        __syncthreads();
    }
    return m;
}

__global__ void __launch_bounds__(512)
nms_smem_kernel(const float4* __restrict__ box, const float* __restrict__ score, const int32_t* __restrict__ count,
                int stride, float thr, int limit, int32_t* __restrict__ keep_idx, int32_t* __restrict__ keep_count, int blockwise) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int prob = blockIdx.x;
    const int n = min(count[prob], stride);
    const int tid = threadIdx.x, T = blockDim.x;
    if (n <= 0) { if (tid == 0) keep_count[prob] = 0; return; }
    const NmsSmem s = nms_carve(smem, stride);
    for (int i = tid; i < n; i += T) {
        s.key[i] = score ? score_key(score[(size_t)prob * stride + i], i) : (unsigned long long)(unsigned)(n - 1 - i);
        s.rank[i] = 0;
    }
    __syncthreads();
    const int m = nms_core(s, box + (size_t)prob * stride, n, thr, limit, keep_idx + (size_t)prob * stride, nullptr, nullptr, blockwise != 0);
    if (tid == 0) keep_count[prob] = m;
}

// K1 + K2 fused for the whole-path call: a CTA decodes the cells of one (image, part), compacts the candidates
// into SHARED memory (never to HBM) and suppresses them right there; what leaves the kernel is the list of surviving
// root CELLS in visiting order.  All six values of a cell are loaded up front so the CTA pays one HBM round trip.
// PERSISTENT: the grid is at most what is resident at once beside the arg-max ring, and every CTA strides over the
// (image, part) lists.  A programmatic dependent is only launched once EVERY CTA of its primary has triggered —
// with one CTA per list a big batch runs in several waves, and whatever follows in the stream (the arg-max kernel)
// could not start before the last wave had; with a resident grid the trigger fires at once and this kernel's whole
// run hides under the arg-max stream (cfg3, 1024 dense images: the step went from 359 us to the arg-max's own time).
template <typename T>
__global__ void __launch_bounds__(512, 3)
decode_nms_kernel(const T* __restrict__ head, Geom g, int n_parts, float det_thr, float nms_thr,
                  int32_t* __restrict__ keep_cell, int32_t* __restrict__ keep_count, int pdl) {
    extern __shared__ __align__(128) unsigned char smem[];
    // pdl & 2: launched as a programmatic dependent itself (of the previous call's tree parse, or of
    // whatever kernel produced `head`): it may have become resident early, so it must wait before it
    // reads anything.  pdl & 1: then release the arg-max kernel, which needs nothing from this one.
    tl_mark(g, TL_START);
    if (pdl & PDL_WAIT_START) pdl_wait();
    tl_mark(g, TL_WAITED);
    if (pdl & PDL_TRIGGER) pdl_launch_dependents();
    __shared__ int warp_tot[16];
    __shared__ int base_s;
    float4* ubox = reinterpret_cast<float4*>(smem);                         // [HW] candidate boxes, cell order
    int32_t* ucell = reinterpret_cast<int32_t*>(ubox + g.HW);               // [HW]
    const NmsSmem s = nms_carve(reinterpret_cast<unsigned char*>(ucell + ((g.HW + 3) & ~3)), g.HW);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_lists = g.B * n_parts;
    for (int item = blockIdx.x; item < n_lists; item += gridDim.x) {
        const int b = item / n_parts, k = item - b * n_parts;
        const T* img = head + (size_t)b * g.img_stride;
        if (tid == 0) base_s = 0;
        for (int i = tid; i < g.HW; i += blockDim.x) s.rank[i] = 0;
        __syncthreads();
        for (int c0 = 0; c0 < g.HW; c0 += blockDim.x) {
            const int c = c0 + tid;
            float d = 0.0f;
            float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
            bool hit = false;
            if (c < g.HW) {
                d = delta_at(img, g, k, c);
                bx = box_at(img, g, k, c);                       // loads issued before d is tested
                hit = d > det_thr;                               // strict, datatest.py:89
            }
            const unsigned bal = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) warp_tot[warp] = __popc(bal);
            __syncthreads();
            int off = base_s, total = 0;
            for (int wi = 0; wi < (int)(blockDim.x >> 5); ++wi) {
                const int t = warp_tot[wi];
                if (wi < warp) off += t;
                total += t;
            }
            if (hit) {
                const int slot = off + __popc(bal & ((1u << lane) - 1u));
                ucell[slot] = c;
                ubox[slot] = bx;
                s.key[slot] = score_key(d, slot);                // ties: larger candidate index (= larger cell) first
            }
            __syncthreads();
            if (tid == 0) base_s += total;
            __syncthreads();
        }
        const int n = base_s;
        const size_t list = (size_t)item * g.HW;
        int m = 0;
        if (n > 0) m = nms_core(s, ubox, n, nms_thr, 0, keep_cell + list, ucell, nullptr, (pdl & NMS_BLOCKWISE) != 0, false);
        if (tid == 0) keep_count[item] = m;
        __syncthreads();                                         // the scratch is reused by this CTA's next list
    }
    // overlapped calls (PPN_FLAG_INPUT_COMPLETE): this kernel started without waiting for the
    // previous call's tree parse; it must not COMPLETE before it, so that "the arg-max kernel
    // completed" (which waits for us) still implies "everything of the previous call completed"
    tl_mark(g, TL_END);
    if (tid == 0 && (pdl & PDL_WAIT_END)) pdl_wait();
}

// Lists longer than PPN_MAX_CELLS: no bitmask; the CTA visits boxes in order and, for every box
// still alive, marks the later boxes it suppresses.  The visiting order lives in keep_idx itself
// (slot m <= i is only overwritten after order[i] has been consumed) with the sign bit as the
// "suppressed" flag, so no extra workspace is needed.
__global__ void __launch_bounds__(1024)
nms_global_kernel(const float4* __restrict__ box, const float* __restrict__ score, const int32_t* __restrict__ count,
                  int stride, float thr, int limit, int32_t* __restrict__ keep_idx, int32_t* __restrict__ keep_count) {
    const int prob = blockIdx.x;
    const int n = min(count[prob], stride);
    const int tid = threadIdx.x, T = blockDim.x;
    int32_t* out = keep_idx + (size_t)prob * stride;     // doubles as order[] | dead bit
    const float4* pbox = box + (size_t)prob * stride;
    const float* psc = score ? score + (size_t)prob * stride : nullptr;
    __shared__ int m_s;
    if (n <= 0) { if (tid == 0) keep_count[prob] = 0; return; }
    for (int i = tid; i < n; i += T) {
        int rank = i;
        if (psc) {
            const unsigned long long mine = score_key(psc[i], i);
            rank = 0;
            for (int j = 0; j < n; ++j) rank += (score_key(psc[j], j) > mine);
        }
        out[rank] = i;
    }
    if (tid == 0) m_s = 0;
    __syncthreads();
    for (int i = 0; i < n; ++i) {
        const int oi = out[i];
        if (oi < 0) continue;                        // uniform: flags are written before a barrier
        const float4 bi = pbox[oi];
        const float ai = box_area(bi);
        __syncthreads();                             // everyone has read out[i] before slot m_s <= i is reused
        if (tid == 0) out[m_s] = oi;
        for (int j = i + 1 + tid; j < n; j += T) {
            const int oj = out[j];
            if (oj >= 0) {
                const float4 bj = pbox[oj];
                if (suppresses(bj, box_area(bj), bi, ai, thr, thr > 0.0f)) out[j] = oj | (int)0x80000000;
            }
        }
        __syncthreads();
        if (tid == 0) m_s += 1;
        __syncthreads();
        if (limit > 0 && m_s >= limit) break;
    }
    if (tid == 0) keep_count[prob] = m_s;
}

// =========================================================================================
// K4 — tree parse, one CTA per image
// =========================================================================================
// resp, conf (adjacent channel groups: ONE contiguous range) and the image's arg-max map are
// staged in shared memory by two bulk copies (TMA) on one mbarrier — a single HBM round trip —
// so each dependent limb step costs shared-memory reads instead of HBM ones.  The kernel is a
// latency chain, so the chain is kept short:
//   * window index -> (dy - off_h, dx - off_w) comes from a shared-memory table, the walk keeps
//     (row, col) as state: no integer division on the dependent path;
//   * when the track orders form a tree (every part has one limb and one predecessor — checked on
//     the host), the chains of a root are walked by DIFFERENT threads: they write identical
//     values where they share a prefix, and the critical path is the longest chain (7 steps for
//     the reference skeleton) instead of the sum (25);
//   * the write-out is one (human, part) pair per thread, so the scattered x/y/w/h reads of the
//     boxes are in flight together and the stores are contiguous.
// All surviving roots of the image are handled in one pass (positions for up to H*W roots fit in
// shared memory).  `use_tma` = 0 (byte ranges not 16-byte multiples): cooperative loads.
constexpr int kMaxDyxTable = 2048;

// launch-chain bits shared by the tree parse and the fused parse kernel (see parse_fused_kernel's header comment)
enum : int {
    FUSED_GUARD = 8,           // poll sync[0] >= seq before the early trigger
    FUSED_TRIGGER_EARLY = 16,  // launch_dependents before the wait (after the guard)
    FUSED_PUBLISH = 32,        // last CTA publishes seq + 1
    FUSED_WAIT_TOP = 64,       // wait for the previous kernel before reading ANYTHING (the decode planes are its output)
};

__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}


__device__ __forceinline__ int fast_div(int x, uint32_t magic) {      // exact for 0 <= x < 65536
    return magic ? (int)__umulhi((unsigned)x, magic) : x;
}

// kStaged: resp/conf live in shared memory (plain LDS) — otherwise they are read from the head tensor
// through the read-only path.  A compile-time switch, so neither case pays for generic addressing.
template <bool kStaged, typename HT>
__device__ __forceinline__ float delta_lookup(const HT* resp, const HT* conf, int at) {
    if (kStaged) return __fmul_rn(widen(resp[at]), widen(conf[at]));
    return __fmul_rn(ldf(resp + at), ldf(conf + at));
}

template <bool kStaged, typename HT>
__device__ __forceinline__ void walk_chain(const ChainTable& ch, int cidx, int root, const Geom& g, float thr,
                                           const HT* s_resp, const HT* s_conf, const uint16_t* s_amax,
                                           const int32_t* s_dyx, bool use_tab, int16_t* my_pos) {
    int ih = fast_div(root, g.magic_W), iw = root - ih * g.W;
    for (int q = ch.off[cidx]; q < ch.off[cidx + 1]; ++q) {
        const int ei = ch.limb[q], t = ch.part[q];
        const int a = s_amax[ei * g.HW + ih * g.W + iw];
        int jh, jw;
        if (use_tab) {
            const int d = s_dyx[a];
            jh = ih + (d >> 16);
            jw = iw + (int)(int16_t)(d & 0xffff);
        } else {
            const int dy = a / g.sW, dx = a - dy * g.sW;
            jh = ih + dy - g.off_h;
            jw = iw + dx - g.off_w;
        }
        if (jh < 0 || jw < 0 || jh >= g.H || jw >= g.W) break;                         // datatest.py:118
        const int j = jh * g.W + jw;
        if (delta_lookup<kStaged, HT>(s_resp, s_conf, t * g.HW + j) < thr) break;          // datatest.py:121
        my_pos[t] = (int16_t)j;
        ih = jh;
        iw = jw;
    }
}

template <bool kStaged, typename HT>
__global__ void __launch_bounds__(1024)
tree_parse_kernel(const HT* __restrict__ head, Geom g, ChainTable ch, float thr, int min_kp, int n_parts,
                  const uint16_t* __restrict__ amax, const int32_t* __restrict__ cand_cell,
                  const int32_t* __restrict__ keep_idx, const int32_t* __restrict__ keep_count,
                  int32_t* __restrict__ h_count, int32_t* __restrict__ h_root, int32_t* __restrict__ h_cell,
                  float* __restrict__ h_score, float4* __restrict__ h_box, int R, int use_tma, int stage_all, int pdl,
                  int* __restrict__ sync, int seq, int xywh_parts) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int KHW = g.K * g.HW;
    // staged channel groups: 0 = none (big grids: the walk reads resp/conf through L2 and the CTA
    // stays light enough to sit beside the arg-max ring), 2 = resp, conf, 6 = also x, y, w, h
    const int n_groups = stage_all;
    HT* s_planes = reinterpret_cast<HT*>(smem);                                          // [n_groups][K*HW]
    uint16_t* s_amax = reinterpret_cast<uint16_t*>(smem + ((((size_t)n_groups * KHW * sizeof(HT)) + 15) & ~(size_t)15));  // [E*HW] (+pad)
    int32_t* s_root = reinterpret_cast<int32_t*>(s_amax + (((size_t)g.E * g.HW + 7) & ~(size_t)7));  // [HW]
    int32_t* s_slot = s_root + g.HW;                                                   // [HW]
    int32_t* s_dyx = s_slot + g.HW;                                                    // [S] if small
    int16_t* s_pos = reinterpret_cast<int16_t*>(s_dyx + (g.S <= kMaxDyxTable ? g.S : 0));   // [HW][K]
    // crowded images: the x / y / w / h planes of `xywh_parts` parts at a time, [4][xywh_parts][HW] (see the write-out)
    HT* s_xywh = reinterpret_cast<HT*>((reinterpret_cast<uintptr_t>(s_pos) + (size_t)g.HW * g.K * 2 + 15) & ~(uintptr_t)15);   // 16-byte aligned
    __shared__ __align__(8) uint64_t bar;
    __shared__ int warp_tot[32];
    __shared__ int base_s;

    const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const bool use_tab = g.S <= kMaxDyxTable;
    const uint32_t bytes_planes = (uint32_t)n_groups * KHW * (uint32_t)sizeof(HT), bytes_am = (uint32_t)g.E * g.HW * 2u;

    // PERSISTENT: the grid is at most what is resident at once and every CTA strides over the images (see
    // decode_nms_kernel).  Overlapped calls: like the fused parse kernel, trigger at the very top — once the previous
    // call's tree parse has been SEEN complete (it read the workspace set the next call's kernels will write).
    tl_mark(g, TL_START);
    if (pdl & FUSED_GUARD) {
        if (tid == 0) while (ld_acquire(sync) < seq) __nanosleep(200);
        __syncthreads();
    }
    if (pdl & FUSED_TRIGGER_EARLY) pdl_launch_dependents();
    if (use_tma && tid == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
    }
    if (use_tab)
        for (int a = tid; a < g.S; a += T) {
            const int dy = a / g.sW, dx = a - dy * g.sW;
            s_dyx[a] = ((dy - g.off_h) << 16) | ((dx - g.off_w) & 0xffff);
        }
    __syncthreads();
    uint32_t parity = 0;
    bool first = true;
    for (int b = blockIdx.x; b < g.B; b += gridDim.x, parity ^= 1u) {
        const HT* img = head + (size_t)b * g.img_stride;
        const HT* s_resp = kStaged ? s_planes : img;                   // shared when kStaged, else the head tensor
        const HT* s_conf = s_resp + KHW;
        const uint16_t* am = amax + (size_t)b * g.E * g.HW;

        // ---- prologue: nothing here depends on the kernels before this one -----------------------
        if (use_tma) {
            if (tid == 0) {
                mbar_arrive_expect_tx(&bar, bytes_planes + bytes_am);
                if (bytes_planes) bulk_g2s(s_planes, img, bytes_planes, &bar);
            }
        } else {
            for (int i = tid; i < n_groups * KHW; i += T) s_planes[i] = __ldg(img + i);
        }
        if (tid == 0) base_s = 0;
        // ---- from here on we read what the arg-max and decode+NMS kernels wrote ---------------------
        if (first) {
            if (pdl & PDL_WAIT_START) pdl_wait();
            tl_mark(g, TL_WAITED);
            if (pdl & PDL_TRIGGER) pdl_launch_dependents();      // the NEXT call's decode+NMS may become resident
            first = false;
        }
        if (use_tma) {
            if (tid == 0 && bytes_am) bulk_g2s(s_amax, am, bytes_am, &bar);
        } else {
            for (int i = tid; i < g.E * g.HW; i += T) s_amax[i] = am[i];
        }
        const int n_keep = min(keep_count[(size_t)b * n_parts], g.HW);
        // What is not staged is gathered cell by cell in the write-out.  For a crowded image (roots on
        // more than 3/8 of the cells) have the L2 stream the rest of the image's decode block in now,
        // as one contiguous read, so that those gathers are L2 hits instead of scattered DRAM sectors
        // (dense-crowd config: tree parse 111 -> 96 us); for sparse images it would only add traffic.
        const bool crowded = n_keep * 8 >= g.HW * 3;
        if (use_tma && tid == 0 && n_groups < 6 && crowded)
            bulk_prefetch_l2(img + (size_t)n_groups * KHW, (uint32_t)(6 - n_groups) * KHW * (uint32_t)sizeof(HT));
        const int32_t* keep = keep_idx + (size_t)b * n_parts * g.HW;
        const int32_t* cells = cand_cell ? cand_cell + (size_t)b * n_parts * g.HW : nullptr;

        // ---- 1. roots and cleared positions (the loads fly with the bulk copies) --------------------
        for (int i = tid; i < n_keep * g.K; i += T) s_pos[i] = -1;
        for (int r = tid; r < n_keep; r += T) s_root[r] = cells ? cells[keep[r]] : keep[r];
        __syncthreads();                          // also: cooperative loads visible
        for (int r = tid; r < n_keep; r += T) s_pos[r * g.K] = (int16_t)s_root[r];
        if (use_tma) mbar_wait(&bar, parity);     // on every path: never go on under an in-flight copy
        if (n_keep == 0) {
            if (tid == 0) h_count[b] = 0;
            __syncthreads();
            continue;
        }
        __syncthreads();

        // ---- 2. walk: one thread per (chain, root) when the track orders are a tree -----------------
        const int n_pad = (n_keep + 31) & ~31;    // whole warps share a chain: uniform chain-table reads
        const int n_par = ch.parallel_ok ? ch.n_chains : 1;
        for (int item = tid; item < n_par * n_pad; item += T) {
            const int cidx = item / n_pad, r = item - cidx * n_pad;
            if (r < n_keep) {
                int16_t* my_pos = s_pos + r * g.K;
                if (ch.parallel_ok) {
                    walk_chain<kStaged, HT>(ch, cidx, s_root[r], g, thr, s_resp, s_conf, s_amax, s_dyx, use_tab, my_pos);
                } else {
                    for (int c = 0; c < ch.n_chains; ++c)
                        walk_chain<kStaged, HT>(ch, c, s_root[r], g, thr, s_resp, s_conf, s_amax, s_dyx, use_tab, my_pos);
                }
            }
        }
        __syncthreads();

        // ---- 3. humans with enough parts take consecutive output slots, in root order ---------------
        for (int r0 = 0; r0 < n_keep; r0 += T) {
            const int r = r0 + tid;
            bool valid = false;
            if (r < n_keep) {
                int present = 0;
                for (int t = 1; t < g.K; ++t) present += (s_pos[r * g.K + t] >= 0);
                valid = min_kp <= present;                                          // datatest.py:129
            }
            const unsigned bal = __ballot_sync(0xffffffffu, valid);
            if (lane == 0) warp_tot[warp] = __popc(bal);
            __syncthreads();
            int off = base_s, total = 0;
            for (int wi = 0; wi < (T >> 5); ++wi) {
                const int v = warp_tot[wi];
                if (wi < warp) off += v;
                total += v;
            }
            const int slot = off + __popc(bal & ((1u << lane) - 1u));
            if (r < n_keep) s_slot[r] = (valid && slot < R) ? slot : -1;
            __syncthreads();
            if (tid == 0) base_s += total;
        }
        __syncthreads();

        // ---- 4. write-out ------------------------------------------------------------------------------
        // Crowded image (dense crowds: a human on nearly every cell): gathering x, y, w, h of every (human, part)
        // pair cell by cell costs a 32-byte L2 sector per 4-byte value — 16 K sectors per image, and every one
        // of them competes with the arg-max stream for L2 throughput (measured at cfg3: the arg-max kernel beside
        // this one took 307 us instead of 222).  Instead the four planes of a few parts at a time are brought into
        // shared memory with coalesced loads (exactly the bytes the head tensor holds, once) and read from there.
        if (crowded && xywh_parts > 0 && n_groups < 6) {
            const int P = xywh_parts, PHW = P * g.HW;
            constexpr int kVec = 16 / (int)sizeof(HT);            // elements per 128-bit load
            const bool vec_ok = (g.HW % kVec) == 0 && (g.img_stride % kVec) == 0 && (reinterpret_cast<uintptr_t>(head) & 15) == 0;
            for (int t0 = 0; t0 < g.K; t0 += P) {
                const int np = min(P, g.K - t0), n_el = np * g.HW;
                if (vec_ok) {                                     // the four planes' loads of a thread are in flight together
                    const int n_vec = n_el / kVec;
                    for (int j = tid; j < n_vec; j += T) {
                        uint4 v[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            v[q] = __ldg(reinterpret_cast<const uint4*>(img + (size_t)(2 + q) * KHW + (size_t)t0 * g.HW) + j);
#pragma unroll
                        for (int q = 0; q < 4; ++q) reinterpret_cast<uint4*>(s_xywh + q * PHW)[j] = v[q];
                    }
                } else {
                    for (int q = 0; q < 4; ++q)
                        for (int j = tid; j < n_el; j += T) s_xywh[q * PHW + j] = __ldg(img + (size_t)(2 + q) * KHW + (size_t)t0 * g.HW + j);
                }
                __syncthreads();
                const uint32_t magic_np = np <= 1 ? 0u : (uint32_t)(((1ull << 32) + np - 1) / np);   // exact pi / np below 65536
                for (int pi = tid; pi < n_keep * np; pi += T) {
                    const int r = fast_div(pi, magic_np), tt = pi - r * np, t = t0 + tt;
                    const int sl = s_slot[r];
                    if (sl < 0) continue;
                    const int c = s_pos[r * g.K + t];
                    float score = 0.0f;
                    float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (c >= 0) {
                        const int at = t * g.HW + c, a2 = tt * g.HW + c;
                        const int h = fast_div(c, g.magic_W), w = c - h * g.W;
                        score = delta_lookup<kStaged, HT>(s_resp, s_conf, at);
                        box = box_from(widen(s_xywh[a2]), widen(s_xywh[PHW + a2]), widen(s_xywh[2 * PHW + a2]),
                                       widen(s_xywh[3 * PHW + a2]), h, w, g);
                    }
                    const size_t human = (size_t)b * R + sl, o = human * g.K + t;
                    if (t == 0) h_root[human] = c;
                    h_cell[o] = c;
                    h_score[o] = score;
                    h_box[o] = box;
                }
                __syncthreads();
            }
        }
        // otherwise one (human, part) pair per thread and step, four steps in flight
        const int n_pairs = (crowded && xywh_parts > 0 && n_groups < 6) ? 0 : n_keep * g.K;
        for (int p0 = tid; p0 < n_pairs; p0 += 4 * T) {
            int cc[4], tt[4], ss[4];
            float xs[4], ys[4], ws[4], hs[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int pair = p0 + u * T;
                cc[u] = -2;                                       // -2: nothing to write
                if (pair < n_pairs) {
                    const int r = fast_div(pair, g.magic_K), t = pair - r * g.K;
                    const int sl = s_slot[r];
                    if (sl >= 0) {
                        cc[u] = s_pos[pair];
                        tt[u] = t;
                        ss[u] = sl;
                        if (cc[u] >= 0) {
                            const int at = t * g.HW + cc[u];
                            if (n_groups == 6) {
                                xs[u] = widen(s_planes[2 * KHW + at]); ys[u] = widen(s_planes[3 * KHW + at]);
                                ws[u] = widen(s_planes[4 * KHW + at]); hs[u] = widen(s_planes[5 * KHW + at]);
                            } else {
                                xs[u] = ldf(img + (size_t)2 * KHW + at); ys[u] = ldf(img + (size_t)3 * KHW + at);
                                ws[u] = ldf(img + (size_t)4 * KHW + at); hs[u] = ldf(img + (size_t)5 * KHW + at);
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (cc[u] == -2) continue;
                const int c = cc[u];
                float score = 0.0f;
                float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
                if (c >= 0) {
                    const int at = tt[u] * g.HW + c;
                    const int h = fast_div(c, g.magic_W), w = c - h * g.W;
                    score = delta_lookup<kStaged, HT>(s_resp, s_conf, at);
                    box = box_from(xs[u], ys[u], ws[u], hs[u], h, w, g);
                }
                const size_t human = (size_t)b * R + ss[u], o = human * g.K + tt[u];
                if (tt[u] == 0) h_root[human] = c;
                h_cell[o] = c;
                h_score[o] = score;
                h_box[o] = box;
            }
        }
        if (tid == 0) h_count[b] = base_s;
        __syncthreads();                          // the shared arrays are reused by this CTA's next image
    }
    tl_mark(g, TL_END);
    // ---- the last CTA publishes this call's sequence number (see parse_fused_kernel) ---------------------
    if (pdl & FUSED_PUBLISH) {
        __syncthreads();
        if (tid == 0 && atomicAdd(sync + 1, 1) == (int)gridDim.x - 1) {
            sync[1] = 0;
            __threadfence();
            atomicMax(sync, seq + 1);
        }
    }
}

// =========================================================================================
// K124 — decode + NMS + tree parse in ONE kernel, one CTA per image (the whole-path call's default)
// =========================================================================================
// Everything the parse needs besides the arg-max map — the root candidates, their NMS, delta of
// every (part, cell) — does not depend on the limb arg-max, so it is this kernel's PROLOGUE: the
// kernel is launched as a programmatic dependent of the arg-max kernel, becomes resident beside it
// at once, decodes and suppresses in shared memory while the arg-max streams the limb block, and
// only then executes griddepcontrol.wait.  What is left after the wait is the walk and the
// write-out.  Per call that is two launches (K3, K124) and no root lists in HBM.
//
// Consecutive overlapped calls (PPN_FLAG_INPUT_COMPLETE): K124(i) lets the NEXT call's arg-max
// K3(i+1) be launched as soon as K124(i) is resident — long before K3(i) ends — so K3(i+1)'s CTAs
// take over the SMs one by one as K3(i)'s CTAs exit and the limb stream never pauses between calls.
// Two things make that safe:
//  * K3(i+1) writes the arg-max buffer and draws from the ticket counters that call i-1 used.
//    K124(i) therefore triggers only after it has SEEN K124(i-1) complete: the last CTA of every
//    K124 publishes its sequence number (`sync[0]`, monotonic), and K124(i) polls it before
//    griddepcontrol.launch_dependents.  K124(i-1) complete implies K3(i-1) complete (it waited for it).
//    The poll cannot deadlock: K124(i) is only launched once every CTA of K3(i) has started, K3(i)
//    only once every CTA of K124(i-1) was resident, and K124(i-1) waits only for K3(i-1), all of
//    whose CTAs had started before K124(i-1) was launched.
//  * completion stays transitive: K3(i+1) waits at its END for K124(i) (its programmatic primary),
//    K124(i+1) waits for K3(i+1) — calls complete in order.
// Sequence numbers are host state and would be frozen by stream capture; under capture (and without
// the flag) the kernel triggers only AFTER its wait, which bounds the overlap to two calls without
// any flag (K3(i+1) launched => K3(i) complete => K124(i-1) complete).
struct FusedSmem { uint32_t delta, root, dyx, uni, amax, slot, estart, pmask, pos, total; };

__host__ __device__ inline FusedSmem fused_layout(const Geom& g, bool staged) {
    FusedSmem l;
    uint32_t off = 0;
    l.delta = off; off += staged ? (uint32_t)g.K * g.HW * 4u : 0u;
    l.root = off;  off += (uint32_t)g.HW * 4u;
    l.dyx = off;   off += g.S <= 2048 ? (uint32_t)g.S * 4u : 0u;
    off = (off + 15u) & ~15u;
    l.uni = off;                                               // NMS scratch, later reused by the walk
    const uint32_t nms = (uint32_t)g.HW * 16u + (((uint32_t)g.HW + 3u) & ~3u) * 4u + (uint32_t)nms_bytes_per_list(g.HW);
    l.amax = l.uni;
    l.slot = l.amax + ((((uint32_t)g.E * g.HW * 2u) + 15u) & ~15u);
    l.estart = l.slot + (uint32_t)g.HW * 4u;
    l.pmask = l.estart + (uint32_t)g.HW * 4u;
    l.pos = l.pmask + (uint32_t)g.HW * 4u;
    const uint32_t walk = (l.pos - l.uni) + ((((uint32_t)g.HW * g.K * 2u) + 15u) & ~15u);
    l.total = l.uni + (nms > walk ? nms : walk);
    return l;
}

// Optional second output of the fused kernel: the dense (human, part) entry buffer of the multi-GPU
// gather (layout: see "pack" below), written straight from shared memory — no pack kernel, no pass
// over the fixed-stride arrays.  An image's entries are contiguous and ordered (human, part); images
// take their place with one atomicAdd on header[0] (which the caller zeroes before the launch), so
// the ORDER of the images' blocks is arbitrary and header.start[b] says where image b begins.
struct DenseOut {
    int32_t* header;       // nullptr: no dense output.  Always LOCAL memory: the cursor is an atomic
    int32_t* rheader;      // nullptr, or the header of the buffer the entries go to when that is ANOTHER buffer — e.g. the
                           // gather root's, mapped over NVLink: the per-image table is then stored there as well, and
                           // idcell / score / box below point into that buffer (plain stores, nothing is read back)
    uint32_t* idcell;
    float* score;
    float4* box;
    int32_t cap;
    int32_t skip_slots;    // 1: the fixed-stride arrays (root_cell, part_*) need not be written; count[] still is
    int32_t B_total, b0;   // the launch covers images [b0, b0 + gridDim.x) of a batch of B_total (header indexing)
};

template <bool kStaged, typename HT>
__global__ void __launch_bounds__(512, 3)
parse_fused_kernel(const HT* __restrict__ head, Geom g, ChainTable ch, float det_thr, float nms_thr, int min_kp,
                   const uint16_t* __restrict__ amax, int32_t* __restrict__ h_count, int32_t* __restrict__ h_root,
                   int32_t* __restrict__ h_cell, float* __restrict__ h_score, float4* __restrict__ h_box, int R,
                   int pdl, int* __restrict__ sync, int seq, DenseOut dense) {
    extern __shared__ __align__(128) unsigned char smem[];
    const FusedSmem L = fused_layout(g, kStaged);
    float* s_delta = reinterpret_cast<float*>(smem + L.delta);                  // [K*HW] resp*conf (kStaged)
    int32_t* s_root = reinterpret_cast<int32_t*>(smem + L.root);                // [HW] surviving root cells
    int32_t* s_dyx = reinterpret_cast<int32_t*>(smem + L.dyx);                  // [S]
    float4* ubox = reinterpret_cast<float4*>(smem + L.uni);                     // NMS phase: candidate boxes,
    int32_t* ucell = reinterpret_cast<int32_t*>(ubox + g.HW);                   //   their cells,
    const NmsSmem s = nms_carve(reinterpret_cast<unsigned char*>(ucell + ((g.HW + 3) & ~3)), g.HW);   // sort + mask
    uint16_t* s_amax = reinterpret_cast<uint16_t*>(smem + L.amax);              // walk phase (same bytes): [E*HW]
    int32_t* s_slot = reinterpret_cast<int32_t*>(smem + L.slot);                // [HW]
    int32_t* s_estart = reinterpret_cast<int32_t*>(smem + L.estart);            // [HW] first dense entry of a human
    uint32_t* s_pmask = reinterpret_cast<uint32_t*>(smem + L.pmask);            // [HW] present parts of a human (K <= 32)
    int16_t* s_pos = reinterpret_cast<int16_t*>(smem + L.pos);                  // [HW][K]
    __shared__ int warp_tot[16];
    __shared__ int warp_ent[16];
    __shared__ int base_s;
    __shared__ int ebase_s;
    __shared__ int n_keep_s;

    const int b = blockIdx.x;
    const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int KHW = g.K * g.HW;
    const HT* img = head + (size_t)b * g.img_stride;
    const bool use_tab = g.S <= kMaxDyxTable;

    tl_mark(g, TL_START);
    if (pdl & FUSED_WAIT_TOP) pdl_wait();       // fused network head: resp/conf/x/y/w/h are the previous kernel's output
    // ---- let the next call's arg-max be launched (see the header comment): it only queues behind
    //      this call's arg-max, so the earlier the better ---------------------------------------------
    if (pdl & FUSED_GUARD) {
        if (tid == 0) while (ld_acquire(sync) < seq) __nanosleep(200);
        __syncthreads();
    }
    if (pdl & FUSED_TRIGGER_EARLY) pdl_launch_dependents();
    // resp and conf of every part are read below anyway (delta staging / the walk): ask the L2 for them now,
    // as one contiguous read, so that those loads find them there instead of each paying a DRAM round trip
    if (tid == 0 && ((size_t)2 * g.K * g.HW * sizeof(HT)) % 16 == 0 && (g.img_stride * sizeof(HT)) % 16 == 0 &&
        (reinterpret_cast<uintptr_t>(head) & 15) == 0)
        bulk_prefetch_l2(head + (size_t)blockIdx.x * g.img_stride, (uint32_t)2 * g.K * g.HW * (uint32_t)sizeof(HT));

    tl_phase(g, 1);
    // ---- prologue 1: root candidates of part 0, compacted into shared memory (datatest.py:80-92) ----
    if (tid == 0) { base_s = 0; n_keep_s = 0; }
    for (int i = tid; i < g.HW; i += T) s.rank[i] = 0;
    if (use_tab)
        for (int a = tid; a < g.S; a += T) {
            const int dy = a / g.sW, dx = a - dy * g.sW;
            s_dyx[a] = ((dy - g.off_h) << 16) | ((dx - g.off_w) & 0xffff);
        }
    __syncthreads();
    for (int c0 = 0; c0 < g.HW; c0 += T) {
        const int c = c0 + tid;
        float d = 0.0f;
        float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
        bool hit = false;
        if (c < g.HW) {
            d = delta_at(img, g, 0, c);
            bx = box_at(img, g, 0, c);
            hit = d > det_thr;                               // strict, datatest.py:89
        }
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) warp_tot[warp] = __popc(bal);
        __syncthreads();
        int off = base_s, total = 0;
        for (int wi = 0; wi < (T >> 5); ++wi) {
            const int t = warp_tot[wi];
            if (wi < warp) off += t;
            total += t;
        }
        if (hit) {
            const int slot = off + __popc(bal & ((1u << lane) - 1u));
            ucell[slot] = c;
            ubox[slot] = bx;
            s.key[slot] = score_key(d, slot);                // ties: larger candidate index (= larger cell) first
        }
        __syncthreads();
        if (tid == 0) base_s += total;
        __syncthreads();
    }
    tl_phase(g, 2);
    // ---- prologue 2: delta of every (part, cell), one coalesced pass (rt_test.py:130) -----------------
    if (kStaged)
        for (int i = tid; i < KHW; i += T) s_delta[i] = __fmul_rn(ldf(img + i), ldf(img + KHW + i));
    tl_phase(g, 3);
    // ---- prologue 3: NMS of the candidates, survivors' cells in visiting order (datatest.py:93-95) ----
    const int n_cand = base_s;
    if (n_cand > 0) {
        const int m = nms_core(s, ubox, n_cand, nms_thr, 0, s_root, ucell, &g, (pdl & NMS_BLOCKWISE) != 0);
        if (tid == 0) n_keep_s = m;
    }
    __syncthreads();                                          // NMS scratch is dead from here; n_keep_s, s_root visible
    const int n_keep = n_keep_s;
    tl_phase(g, 4);
    // for a crowded image have the L2 stream the x/y/w/h planes in now (one contiguous read): the
    // write-out's scattered gathers are then L2 hits
    if (tid == 0 && n_keep * 8 >= g.HW * 3 && ((size_t)KHW * sizeof(HT)) % 16 == 0 && (g.img_stride * sizeof(HT)) % 16 == 0 &&
        (reinterpret_cast<uintptr_t>(head) & 15) == 0)
        bulk_prefetch_l2(img + (size_t)2 * KHW, (uint32_t)4 * KHW * (uint32_t)sizeof(HT));
    for (int i = tid; i < n_keep * g.K; i += T) s_pos[i] = -1;
    __syncthreads();
    for (int r = tid; r < n_keep; r += T) s_pos[r * g.K] = (int16_t)s_root[r];

    // ---- from here on we read what the arg-max kernel wrote -------------------------------------------
    if (pdl & PDL_WAIT_START) pdl_wait();
    tl_mark(g, TL_WAITED);
    if (pdl & PDL_TRIGGER) pdl_launch_dependents();
    if (n_keep > 0) {
        const uint16_t* am = amax + (size_t)b * g.E * g.HW;    // L2 loads: the map was written while we were resident
        const int n16 = (g.E * g.HW) >> 3;
        if ((reinterpret_cast<uintptr_t>(am) & 15) == 0) {
            const uint4* src = reinterpret_cast<const uint4*>(am);
            uint4* dst = reinterpret_cast<uint4*>(s_amax);
            for (int i = tid; i < n16; i += T) dst[i] = __ldcg(src + i);
            for (int i = (n16 << 3) + tid; i < g.E * g.HW; i += T) s_amax[i] = __ldcg(am + i);
        } else {
            for (int i = tid; i < g.E * g.HW; i += T) s_amax[i] = __ldcg(am + i);
        }
    }
    __syncthreads();

    tl_phase(g, 5);
    if (n_keep > 0) {
        const HT* resp = img;
        const HT* conf = img + KHW;
        // ---- walk: one thread per (chain, root) when the track orders are a tree (datatest.py:103-127) ----
        const int n_pad = (n_keep + 31) & ~31;
        const int n_par = ch.parallel_ok ? ch.n_chains : 1;
        for (int item = tid; item < n_par * n_pad; item += T) {
            const int cidx = item / n_pad, r = item - cidx * n_pad;
            if (r >= n_keep) continue;
            int16_t* my_pos = s_pos + r * g.K;
            const int c_lo = ch.parallel_ok ? cidx : 0, c_hi = ch.parallel_ok ? cidx + 1 : ch.n_chains;
            for (int cc = c_lo; cc < c_hi; ++cc) {
                const int root = s_root[r];
                int ih = fast_div(root, g.magic_W), iw = root - ih * g.W;
                for (int q = ch.off[cc]; q < ch.off[cc + 1]; ++q) {
                    const int ei = ch.limb[q], t = ch.part[q];
                    const int a = s_amax[ei * g.HW + ih * g.W + iw];
                    int jh, jw;
                    if (use_tab) {
                        const int d = s_dyx[a];
                        jh = ih + (d >> 16);
                        jw = iw + (int)(int16_t)(d & 0xffff);
                    } else {
                        const int dy = a / g.sW, dx = a - dy * g.sW;
                        jh = ih + dy - g.off_h;
                        jw = iw + dx - g.off_w;
                    }
                    if (jh < 0 || jw < 0 || jh >= g.H || jw >= g.W) break;                     // datatest.py:118
                    const int j = jh * g.W + jw, at = t * g.HW + j;
                    const float dl = kStaged ? s_delta[at] : __fmul_rn(ldf(resp + at), ldf(conf + at));
                    if (dl < det_thr) break;                                                   // datatest.py:121
                    my_pos[t] = (int16_t)j;
                    ih = jh;
                    iw = jw;
                }
            }
        }
        __syncthreads();
        tl_phase(g, 6);
        if (tid == 0) { base_s = 0; ebase_s = 0; }
        __syncthreads();
        // ---- humans with enough parts take consecutive output slots, in root order (datatest.py:129);
        //      their dense entries (one per present part) follow one another in the same order ----------
        for (int r0 = 0; r0 < n_keep; r0 += T) {
            const int r = r0 + tid;
            bool valid = false;
            int present = 0;
            unsigned pm = 1u;                                         // the root is always present
            if (r < n_keep) {
                for (int t = 1; t < g.K; ++t) {
                    const bool here = s_pos[r * g.K + t] >= 0;
                    present += here;
                    pm |= (here && t < 32) ? (1u << t) : 0u;
                }
                valid = min_kp <= present;
            }
            const unsigned bal = __ballot_sync(0xffffffffu, valid);
            if (lane == 0) warp_tot[warp] = __popc(bal);
            __syncthreads();
            int off = base_s, total = 0;
            for (int wi = 0; wi < (T >> 5); ++wi) {
                const int v = warp_tot[wi];
                if (wi < warp) off += v;
                total += v;
            }
            const int slot = off + __popc(bal & ((1u << lane) - 1u));
            const bool placed = valid && slot < R;
            const int n_ent = placed ? present + 1 : 0;               // dense entries of this human
            int incl = n_ent;                                         // warp-inclusive scan
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += up;
            }
            if (lane == 31) warp_ent[warp] = incl;
            __syncthreads();
            int eoff = ebase_s, etotal = 0;
            for (int wi = 0; wi < (T >> 5); ++wi) {
                const int ev = warp_ent[wi];
                if (wi < warp) eoff += ev;
                etotal += ev;
            }
            if (r < n_keep) {
                s_slot[r] = placed ? slot : -1;
                s_estart[r] = eoff + incl - n_ent;
                s_pmask[r] = pm;
            }
            __syncthreads();
            if (tid == 0) { base_s += total; ebase_s += etotal; }
        }
        __syncthreads();
        tl_phase(g, 7);
        // ---- the image's place in the dense buffer ---------------------------------------------------
        const bool want_dense = dense.header != nullptr;
        if (want_dense && tid == 0) {
            const int n_ent = ebase_s, B = dense.B_total, gb = dense.b0 + b;
            const int start = atomicAdd(dense.header, n_ent);
            dense.header[2 + gb] = base_s;
            dense.header[2 + B + gb] = n_ent;
            dense.header[2 + 2 * B + gb] = start;
            if (dense.rheader) {
                dense.rheader[2 + gb] = base_s;
                dense.rheader[2 + B + gb] = n_ent;
                dense.rheader[2 + 2 * B + gb] = start;
            }
            if (start + n_ent > dense.cap) dense.header[1] = 1;
            ebase_s = start + n_ent > dense.cap ? -1 : start;           // -1: the image's entries do not fit
        }
        __syncthreads();
        const int e_base = want_dense ? ebase_s : -1;
        const bool slots_out = !(want_dense && dense.skip_slots);
        // ---- write-out: one (human, part) pair per thread and step, two steps in flight --------------
        const int n_pairs = n_keep * g.K;
        for (int p0 = tid; p0 < n_pairs; p0 += 2 * T) {
            int cc[2], tt[2], ss[2], rr[2];
            float xs[2], ys[2], ws[2], hs[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int pair = p0 + u * T;
                cc[u] = -2;                                       // -2: nothing to write
                if (pair < n_pairs) {
                    const int r = fast_div(pair, g.magic_K), t = pair - r * g.K;
                    const int sl = s_slot[r];
                    if (sl >= 0) {
                        cc[u] = s_pos[pair];
                        tt[u] = t;
                        ss[u] = sl;
                        rr[u] = r;
                        if (cc[u] >= 0) {
                            const int at = t * g.HW + cc[u];
                            xs[u] = ldf(img + (size_t)2 * KHW + at); ys[u] = ldf(img + (size_t)3 * KHW + at);
                            ws[u] = ldf(img + (size_t)4 * KHW + at); hs[u] = ldf(img + (size_t)5 * KHW + at);
                        }
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                if (cc[u] == -2) continue;
                const int c = cc[u];
                float score = 0.0f;
                float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
                if (c >= 0) {
                    const int at = tt[u] * g.HW + c;
                    const int h = fast_div(c, g.magic_W), w = c - h * g.W;
                    score = kStaged ? s_delta[at] : __fmul_rn(ldf(resp + at), ldf(conf + at));
                    box = box_from(xs[u], ys[u], ws[u], hs[u], h, w, g);
                }
                if (slots_out) {
                    const size_t human = (size_t)b * R + ss[u], o = human * g.K + tt[u];
                    if (tt[u] == 0) h_root[human] = c;
                    h_cell[o] = c;
                    h_score[o] = score;
                    h_box[o] = box;
                }
                if (e_base >= 0 && c >= 0) {
                    const int r = rr[u];
                    const int e = e_base + s_estart[r] + __popc(s_pmask[r] & ((1u << tt[u]) - 1u));
                    dense.idcell[e] = ((uint32_t)tt[u] << 16) | (uint32_t)c;
                    dense.score[e] = score;
                    dense.box[e] = box;
                }
            }
        }
    } else if (dense.header != nullptr && tid == 0) {                     // no humans: an empty block
        const int B = dense.B_total, gb = dense.b0 + b;
        dense.header[2 + gb] = 0;
        dense.header[2 + B + gb] = 0;
        dense.header[2 + 2 * B + gb] = 0;
        if (dense.rheader) {
            dense.rheader[2 + gb] = 0;
            dense.rheader[2 + B + gb] = 0;
            dense.rheader[2 + 2 * B + gb] = 0;
        }
    }
    if (tid == 0) h_count[b] = n_keep > 0 ? base_s : 0;
    tl_mark(g, TL_END);
    // ---- the last CTA publishes this call's sequence number ------------------------------------------
    if (pdl & FUSED_PUBLISH) {
        __syncthreads();
        // (what a later kernel must not overtake are this kernel's READS of the arg-max map, and those are
        //  long consumed here — no fence per CTA; the one before the flag orders the counter reset)
        if (tid == 0 && atomicAdd(sync + 1, 1) == (int)gridDim.x - 1) {
            sync[1] = 0;
            __threadfence();
            atomicMax(sync, seq + 1);
        }
    }
}

// =========================================================================================
// part centres — what the consumers right after the path read off each box
// =========================================================================================
// datatest.py:200-211 (drawing) and :316-317 (AP-evaluation records) both reduce a part's box to
// its centre, y = (ymin + ymax) / 2, x = (xmin + xmax) / 2 in fp32 (an add and an exact halving).
// One thread per (image, slot, part); slots beyond count[b] and absent parts give (0, 0).
__global__ void __launch_bounds__(256)
part_centres_kernel(const int32_t* __restrict__ count, const int32_t* __restrict__ cell, const float4* __restrict__ box,
                    size_t n, int R, int K, float2* __restrict__ centre) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t human = i / K;
    const int b = (int)(human / R), slot = (int)(human - (size_t)b * R);
    float2 c = make_float2(0.0f, 0.0f);
    if (slot < count[b] && cell[i] >= 0) c = box_centre(box[i]);
    centre[i] = c;
}

// =========================================================================================
// skeleton — drawing primitives of the webcam loop, straight from the packed result
// =========================================================================================
// What draw_humans (datatest.py:162-232, called at rt_test.py:138-145) computes per human in Python, for every
// slot of the batch in one launch:
//   rect     [B, R, 4]    int32  the root box as it is drawn: (xmin, ymin, xmax, ymax) truncated like int() (:177-181)
//   keypoint [B, R, K, 2] fp32   (x, y) = box centre of every present part (:200-202), NaN where absent
//   segment  [B, R, E, 4] fp32   (bx, by, ex, ey) of every limb whose two parts are present (:213-221), NaN else
// One thread per (image, slot, item), item = rect | part k | limb e.  Same fp32 arithmetic as numpy's: an add and
// an exact halving.  Slots beyond count[b] give rect 0 and NaNs.
struct EdgePairs { uint8_t src[256]; uint8_t dst[256]; };

__global__ void __launch_bounds__(256)
skeleton_kernel(const int32_t* __restrict__ count, const int32_t* __restrict__ cell, const float4* __restrict__ box, size_t n,
                int R, int K, int E, EdgePairs edges, int4* __restrict__ rect, float2* __restrict__ keypoint,
                float4* __restrict__ segment) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int per = 1 + K + E;
    const size_t human = i / per;
    const int item = (int)(i - human * per);
    const int b = (int)(human / R), slot = (int)(human - (size_t)b * R);
    const bool live = slot < count[b];
    const float nan = __int_as_float(0x7fc00000);
    const size_t base = human * K;
    auto centre = [&](int k, float& x, float& y) -> bool {
        if (!live || cell[base + k] < 0) return false;
        const float4 bx = box[base + k];
        y = __fmul_rn(__fadd_rn(bx.x, bx.z), 0.5f);
        x = __fmul_rn(__fadd_rn(bx.y, bx.w), 0.5f);
        return true;
    };
    if (item == 0) {
        int4 r = make_int4(0, 0, 0, 0);
        if (live && cell[base] >= 0) {
            const float4 bx = box[base];                               // (ymin, xmin, ymax, xmax)
            r = make_int4(__float2int_rz(bx.y), __float2int_rz(bx.x), __float2int_rz(bx.w), __float2int_rz(bx.z));
        }
        rect[human] = r;
    } else if (item <= K) {
        const int k = item - 1;
        float x, y;
        keypoint[base + k] = centre(k, x, y) ? make_float2(x, y) : make_float2(nan, nan);
    } else {
        const int e = item - 1 - K;
        float bx, by, ex, ey;
        const bool ok = centre(edges.src[e], bx, by) && centre(edges.dst[e], ex, ey);
        segment[human * E + e] = ok ? make_float4(bx, by, ex, ey) : make_float4(nan, nan, nan, nan);
    }
}

// =========================================================================================
// pack — dense pose entries for the multi-GPU gather
// =========================================================================================
// Fixed-stride PPNHumans -> one contiguous buffer of (human, part) ENTRIES, present parts only:
//   header   int32 {total entries, overflow, count[B], entries[B], start[B]}
//   idcell   uint32[cap]  = part id << 16 | cell        (the root, part 0, is always a human's first
//   score    float [cap]                                  entry, so the list delimits itself)
//   box      float4[cap]
// Most humans have a few of K parts, so this is several times smaller than K slots per human.
// Two launches: per-image entry counts, then one CTA per image places its entries behind the
// entries of the images before it (B coalesced loads) and its humans behind one another (scan).
__global__ void __launch_bounds__(256)
pack_count_kernel(const int32_t* __restrict__ count, const int32_t* __restrict__ cell, int R, int K,
                  int32_t* __restrict__ header, int B) {
    __shared__ int red[8];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = min(count[b], R);
    const int32_t* c = cell + (size_t)b * R * K;
    int present = 0;
    for (int i = tid; i < n * K; i += blockDim.x) present += (c[i] >= 0);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) present += __shfl_xor_sync(0xffffffffu, present, o);
    if (lane == 0) red[warp] = present;
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
        for (int wi = 0; wi < (int)(blockDim.x >> 5); ++wi) tot += red[wi];
        header[2 + b] = count[b];
        header[2 + B + b] = tot;
    }
}

__global__ void __launch_bounds__(256)
pack_entries_kernel(const int32_t* __restrict__ count, const int32_t* __restrict__ cell, const float* __restrict__ score,
                    const float4* __restrict__ box, int B, int R, int K, int cap, int32_t* __restrict__ header,
                    uint32_t* __restrict__ e_idcell, float* __restrict__ e_score, float4* __restrict__ e_box) {
    extern __shared__ __align__(16) int s_start[];          // [n + 1] entry offset of every human of the image
    __shared__ int red[8];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n_warps = blockDim.x >> 5;
    const int32_t* per_image = header + 2 + B;
    int before = 0;
    for (int i = tid; i < b; i += blockDim.x) before += per_image[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if (lane == 0) red[warp] = before;
    __syncthreads();
    int off = 0;
    for (int wi = 0; wi < n_warps; ++wi) off += red[wi];
    if (tid == 0) {
        header[2 + 2 * B + b] = off;                        // start[b]: images in order here (the fused kernel: any order)
        if (b == B - 1) {
            const int total = off + per_image[b];
            header[0] = total;
            header[1] = total > cap ? 1 : 0;
        }
    }
    const int n = min(count[b], R);
    const int32_t* c = cell + (size_t)b * R * K;
    // parts per human, one warp per human (lanes = parts, 32 at a time), then an exclusive scan
    for (int h = warp; h < n; h += n_warps) {
        int cnt = 0;
        for (int t0 = 0; t0 < K; t0 += 32) {
            const int t = t0 + lane;
            cnt += __popc(__ballot_sync(0xffffffffu, t < K && c[h * K + t] >= 0));
        }
        if (lane == 0) s_start[h + 1] = cnt;
    }
    __syncthreads();
    if (warp == 0) {                                        // n <= 1024: 32 humans per step
        int carry = 0;
        for (int h0 = 0; h0 < n; h0 += 32) {
            const int h = h0 + lane;
            int v = h < n ? s_start[h + 1] : 0, incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += up;
            }
            if (h < n) s_start[h + 1] = carry + incl;
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) s_start[0] = 0;
    }
    __syncthreads();
    for (int h = warp; h < n; h += n_warps) {
        int base = off + s_start[h];
        for (int t0 = 0; t0 < K; t0 += 32) {
            const int t = t0 + lane;
            const int cc = t < K ? c[h * K + t] : -1;
            const unsigned bal = __ballot_sync(0xffffffffu, cc >= 0);
            const int pos = base + __popc(bal & ((1u << lane) - 1u));
            if (cc >= 0 && pos < cap) {
                const size_t src = ((size_t)b * R + h) * K + t;
                e_idcell[pos] = ((uint32_t)t << 16) | (uint32_t)cc;
                e_score[pos] = score[src];
                e_box[pos] = box[src];
            }
            base += __popc(bal);
        }
    }
}

// =========================================================================================
// launchers
// =========================================================================================
// run `...` with T bound to the head tensor's element type
#define PPN_DISPATCH_HEAD(dtype, ...)                                                        \
    switch (dtype) {                                                                         \
        case HEAD_F32: { using T = float; __VA_ARGS__; } break;                              \
        case HEAD_F16: { using T = __half; __VA_ARGS__; } break;                             \
        case HEAD_BF16: { using T = __nv_bfloat16; __VA_ARGS__; } break;                     \
        default: return cudaErrorInvalidValue;                                               \
    }

// Per-stream device words (the only memory the library ever allocates: 2 KB per device, on the
// first launch — so make the first call outside stream capture):
//   [0..3] two {next ticket, finished CTAs} pairs of the ring kernels, used ALTERNATELY by successive
//          launches on the stream (consecutive arg-max launches may overlap, see K124), zero between
//          uses: the last CTA of a launch resets its pair;
//   [4..5] {published sequence number, finished CTAs} of the fused parse kernel.
// Kernels on different streams get different slots.
constexpr int kTicketSlots = 64;
constexpr int kSlotWords = 8;
struct StreamSlot { cudaStream_t stream = nullptr; unsigned launches = 0; unsigned calls = 0; int published = 0; bool fast_open = false; };
struct DeviceInfo { int* tickets = nullptr; StreamSlot slot[kTicketSlots]; int slots_used = 0;
                    int sms = 0; int smem_optin = 0; size_t tma = 0, tma_multi = 0, tma16[2] = {0, 0}, decode_nms[3] = {0, 0, 0}, ldg = 0, nms = 0,
                           tree[3] = {0, 0, 0}, tree_light[3] = {0, 0, 0}, fused[2][3] = {{0, 0, 0}, {0, 0, 0}}, cluster[3] = {0, 0, 0}; };
static DeviceInfo g_dev[64];

// Properties and per-kernel dynamic-shared-memory opt-ins are per device; one process normally
// drives one GPU, but nothing here assumes it.
static cudaError_t device_info(DeviceInfo** out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    DeviceInfo& d = g_dev[dev];
    if (!d.sms) {
        int sms = 0, optin = 0;
        if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
        if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
        d.smem_optin = optin;
        d.sms = sms;
    }
    *out = &d;
    return cudaSuccess;
}

// First use of a kernel on a device (and whenever it needs more dynamic shared memory than it was
// last granted): raise its limit and ask for the largest shared-memory carveout.  The carveout is
// an SM-wide setting; if the ring kernel were given just enough for itself, no CTA of another
// kernel could become resident beside it and the side-stream overlap in ppn_parse would silently
// serialise (measured: it did).
static std::mutex g_ticket_mu;

// The stream's slot (nullptr when all slots are taken: callers then deal work statically and do
// not overlap calls).  Caller holds no lock.
static cudaError_t slot_for(DeviceInfo* d, cudaStream_t st, StreamSlot** slot, int** words) {
    std::lock_guard<std::mutex> lock(g_ticket_mu);
    if (!d->tickets) {
        cudaError_t e = cudaMalloc(&d->tickets, kTicketSlots * kSlotWords * sizeof(int));
        if (e != cudaSuccess) return e;
        if ((e = cudaMemset(d->tickets, 0, kTicketSlots * kSlotWords * sizeof(int))) != cudaSuccess) return e;
    }
    *slot = nullptr;
    *words = nullptr;
    for (int i = 0; i < d->slots_used; ++i)
        if (d->slot[i].stream == st) { *slot = &d->slot[i]; *words = d->tickets + kSlotWords * i; return cudaSuccess; }
    if (d->slots_used == kTicketSlots) {
        // Every slot is taken: hand over one whose stream has nothing in flight (or no longer exists).  Its device
        // words are at rest then — ticket pairs zero, the published sequence number equal to the host's copy — so
        // the new stream simply continues the numbering.  A busy stream keeps its slot.
        for (int i = 0; i < kTicketSlots; ++i) {
            const cudaError_t q = cudaStreamQuery(d->slot[i].stream);
            if (q == cudaErrorNotReady) continue;
            if (q != cudaSuccess) (void)cudaGetLastError();          // a destroyed stream: clear the error, take the slot
            d->slot[i].stream = st;
            d->slot[i].fast_open = false;
            *slot = &d->slot[i];
            *words = d->tickets + kSlotWords * i;
            return cudaSuccess;
        }
        return cudaSuccess;                                          // all busy: the caller deals work statically
    }
    d->slot[d->slots_used].stream = st;
    *slot = &d->slot[d->slots_used];
    *words = d->tickets + kSlotWords * d->slots_used++;
    return cudaSuccess;
}

// Which half of the caller's workspace the next whole-path call on `st` uses.  Calls can only overlap their
// predecessor on the SAME stream, so alternating per stream is enough; streams without a slot (stream capture, more
// busy streams than slots) alternate on a per-thread counter.
unsigned next_call_parity(cudaStream_t st) {
    static thread_local unsigned t_calls = 0;
    DeviceInfo* d = nullptr;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (device_info(&d) != cudaSuccess || cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone)
        return t_calls++ & 1u;
    StreamSlot* slot = nullptr;
    int* words = nullptr;
    if (slot_for(d, st, &slot, &words) != cudaSuccess || !slot) return t_calls++ & 1u;
    std::lock_guard<std::mutex> lock(g_ticket_mu);
    return slot->calls++ & 1u;
}

// ticket pair for the next ring-kernel launch on `st`
static cudaError_t ticket_for(DeviceInfo* d, cudaStream_t st, int** out) {
    StreamSlot* slot = nullptr;
    int* words = nullptr;
    cudaError_t e = slot_for(d, st, &slot, &words);
    if (e != cudaSuccess) return e;
    *out = slot ? words + 2 * (slot->launches++ & 1u) : nullptr;
    return cudaSuccess;
}

template <typename F>
static cudaError_t ensure_smem(F kernel, size_t want, size_t* have) {
    if (*have != 0 && want <= *have) return cudaSuccess;
    const size_t grant = want > 48 * 1024 ? want : 48 * 1024;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)grant);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e == cudaSuccess) *have = grant;
    return e;
}

// Launch with (pdl = true) or without the programmatic-stream-serialization attribute: with it the
// kernel may begin while the previous kernel in the stream is still running, once every CTA of that
// kernel has executed griddepcontrol.launch_dependents (or exited).
template <typename... KArgs, typename... Args>
static cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                                 Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Items of G matrices are drawn by `grid` persistent CTAs.  With equal items the CTAs finish up to one item apart
// (cfg2: 960 items on 148 CTAs = 6.5 waves, 7 % of the launch is a half-empty last wave).  So all but the last full
// wave are handed out as items of G, and what is left — between one and two waves of work — as items of G/n (n = 4):
// the same code path with fewer of the thread groups busy, and the CTAs finish within a quarter item of one another.
static void plan_tail(ArgmaxPlan* p, long long n_mats, long long grid, int divide) {
    const long long full_items = n_mats / p->G;
    const long long waves = grid > 0 ? full_items / grid : 0;
    p->small_m = divide > 1 && waves >= 2 ? std::max(1, p->G / divide) : p->G;
    p->n_big = p->small_m == p->G ? (int)((n_mats + p->G - 1) / p->G) : (int)((waves - 1) * grid);
    if (p->small_m == p->G) p->n_big = (int)full_items;          // the remainder (< G matrices) is one last item
}

// host-side view of the item partition, for the CPU test that checks it covers every matrix exactly once
void argmax_item_partition(const ArgmaxPlan& p, int n_mats, int* n_items, int (*first_size)(void*, int, int, int), void* ctx) {
    *n_items = item_count(p, n_mats);
    for (int it = 0; it < *n_items; ++it) {
        const int m0 = item_first(p, it);
        first_size(ctx, it, m0, std::min(item_size(p, it), n_mats - m0));
    }
}

// A tail item holds small_m matrices instead of G: it takes G / small_m times the rows per stage, so that a stage
// still carries about the same bytes (and the bulk copies get longer) — a CTA in the tail streams as fast as before.
static void plan_tail_rows(ArgmaxPlan* p, int S, int row_bytes) {
    p->rows_s = p->rows;
    p->chunks_s = p->chunks;
    if (!row_bytes || p->small_m >= p->G) return;
    int max_rows = (int)(p->stage_bytes / ((size_t)row_bytes * p->small_m));
    max_rows = std::max(1, std::min(max_rows, S));
    p->chunks_s = (S + max_rows - 1) / max_rows;
    p->rows_s = (S + p->chunks_s - 1) / p->chunks_s;
    p->chunks_s = (S + p->rows_s - 1) / p->rows_s;
}

bool plan_argmax(const Geom& g, const Tuning& t, int sms, ArgmaxPlan* p) {
    if (g.HW % 4 != 0 || g.HW / 4 > 992) return false;
    p->CV = g.HW / 4;
    const int row_bytes = g.HW * 4;
    int G = t.argmax_threads / p->CV;
    if (G < 1) G = 1;
    while (G > 1 && p->CV * G > 992) --G;
    // thread groups take one matrix each (mode 1: no merge, no barrier) whenever there are several
    // groups; splitting the rows of one matrix over the groups (mode 0) is kept as the alternative —
    // measured equal or slower at every BASELINE shape (profiles/sweep_argmax_*_r1.txt)
    p->split_mats = (t.argmax_split < 0 ? (G > 1) : (t.argmax_split != 0)) ? 1 : 0;
    if (p->split_mats) {
        if (G > 32) G = 32;                               // one producer lane per matrix
        if (G > g.B * g.E) G = g.B * g.E;
    } else if (G > g.S) {
        G = g.S;
    }
    p->G = G;
    plan_tail(p, (long long)g.B * g.E, (long long)sms * (t.argmax_ctas_per_sm < 1 ? 1 : t.argmax_ctas_per_sm), t.argmax_tail_opt);
    p->threads = p->CV * G;
    p->threads_padded = (p->threads + 31) & ~31;
    const int per_row = p->split_mats ? row_bytes * G : row_bytes;     // ring bytes per row index
    const int stage_target = t.argmax_stage_bytes > 0 ? t.argmax_stage_bytes
                                                      : ((size_t)g.S * row_bytes <= 64 * 1024 ? 48 * 1024 : 32 * 1024);
    int max_rows = stage_target / per_row;
    if (max_rows < 1) max_rows = 1;
    if (max_rows > g.S) max_rows = g.S;
    p->chunks = (g.S + max_rows - 1) / max_rows;
    p->rows = (g.S + p->chunks - 1) / p->chunks;
    p->chunks = (g.S + p->rows - 1) / p->rows;
    p->stage_bytes = (uint32_t)(((size_t)p->rows * per_row + 127) & ~(size_t)127);
    plan_tail_rows(p, g.S, p->split_mats ? row_bytes : 0);
    p->stages = t.argmax_stages;
    p->dry = t.argmax_dry;
    p->ctas_per_sm = t.argmax_ctas_per_sm < 1 ? 1 : t.argmax_ctas_per_sm;
    p->smem_bytes = (size_t)p->stages * p->stage_bytes + (size_t)2 * p->stages * sizeof(uint64_t) +
                    (size_t)p->stages * sizeof(int) + (p->split_mats ? 0 : (size_t)2 * G * g.HW * sizeof(Partial));
    return true;
}

// Ring plan for a 16-bit head: always the split-matrix mapping, 16-byte vectors of 8 columns; items of G matrices
// with the shrinking tail of plan_tail().
static bool plan_argmax16(const Geom& g, const Tuning& t, int sms, ArgmaxPlan* p) {
    if (g.HW % 8 != 0 || g.HW / 8 > 992) return false;
    p->CV = g.HW / 8;
    const int row_bytes = g.HW * 2;
    int G = t.argmax16_threads / p->CV;
    if (G < 1) G = 1;
    while (G > 1 && p->CV * G > 992) --G;
    if (G > 32) G = 32;
    if (G > g.B * g.E) G = g.B * g.E;
    p->ctas_per_sm = t.argmax_ctas_per_sm < 1 ? 1 : t.argmax_ctas_per_sm;
    p->split_mats = 1;
    p->G = G;
    plan_tail(p, (long long)g.B * g.E, (long long)sms * p->ctas_per_sm, t.argmax_tail_opt);
    p->threads = p->CV * G;
    p->threads_padded = (p->threads + 31) & ~31;
    const int per_row = row_bytes * G;
    int max_rows = t.argmax16_stage_bytes / per_row;
    if (max_rows < 1) max_rows = 1;
    if (max_rows > g.S) max_rows = g.S;
    p->chunks = (g.S + max_rows - 1) / max_rows;
    p->rows = (g.S + p->chunks - 1) / p->chunks;
    p->chunks = (g.S + p->rows - 1) / p->rows;
    p->stage_bytes = (uint32_t)(((size_t)p->rows * per_row + 127) & ~(size_t)127);
    plan_tail_rows(p, g.S, row_bytes);
    p->stages = t.argmax_stages;
    p->dry = t.argmax_dry;
    p->smem_bytes = (size_t)p->stages * p->stage_bytes + (size_t)2 * p->stages * sizeof(uint64_t) + (size_t)p->stages * sizeof(int);
    return true;
}

template <typename T16>
static cudaError_t launch_limb_argmax16(const T16* head, uint16_t* amax, const Geom& g, const Tuning& t, cudaStream_t st,
                                        bool pdl, bool* pdl_used, int pdl_bits, DeviceInfo* d, size_t* have, int32_t* zero2, bool* zeroed) {
    const int n_mats = g.B * g.E;
    ArgmaxPlan p;
    cudaError_t e;
    if (plan_argmax16(g, t, d->sms, &p) && (reinterpret_cast<uintptr_t>(head) & 15) == 0 && (g.img_stride * 2) % 16 == 0 &&
        (g.limb_off * 2) % 16 == 0) {
        size_t budget = (size_t)d->smem_optin / p.ctas_per_sm - (p.ctas_per_sm > 1 ? 1024 : 0);
        {   // honour the per-call cap if a ring of at least two stages fits under it
            const size_t two = p.smem_bytes - (size_t)(p.stages - 2) * (p.stage_bytes + 2 * sizeof(uint64_t) + sizeof(int));
            if (t.argmax_smem_cap > 0 && (size_t)t.argmax_smem_cap < budget && (p.stages < 2 || two <= (size_t)t.argmax_smem_cap))
                budget = (size_t)t.argmax_smem_cap;
        }
        while (p.smem_bytes > budget && p.stages > 2) {
            --p.stages;
            p.smem_bytes -= p.stage_bytes + 2 * sizeof(uint64_t) + sizeof(int);
        }
        if (p.smem_bytes <= budget) {
            int* ticket = nullptr;
            if (t.argmax_dynamic && (e = ticket_for(d, st, &ticket)) != cudaSuccess) return e;
            int grid = d->sms * p.ctas_per_sm;
            const int n_items = item_count(p, n_mats);
            if (grid > n_items) grid = n_items;
            if ((e = ensure_smem(limb_argmax_tma_multi16_kernel<T16>, p.smem_bytes, have)) != cudaSuccess) return e;
            e = launch_kernel(limb_argmax_tma_multi16_kernel<T16>, dim3(grid), dim3(p.threads_padded + 32), p.smem_bytes, st, pdl,
                              head, amax, g, p, pdl_bits, ticket, zero2);
            if (pdl_used) *pdl_used = pdl;
            if (zeroed) *zeroed = zero2 != nullptr;
            return e;
        }
    }
    dim3 grid(n_mats, (g.HW + 255) / 256);
    limb_argmax_generic_kernel<T16><<<grid, 256, 0, st>>>(head, amax, g);
    return cudaGetLastError();
}

// Cluster kernel for tiny batches: taken when the matrices would occupy at most half of the SMs with one CTA
// each (argmax.cluster: -1 auto, 0 never, n > 1 forces clusters of n).
static cudaError_t try_launch_argmax_cluster(const void* head_v, uint16_t* amax, const Geom& g, const Tuning& t, cudaStream_t st,
                                             bool pdl, int pdl_bits, DeviceInfo* d, int32_t* zero2, bool* done) {
    *done = false;
    const int n_mats = g.B * g.E;
    if (t.argmax_cluster == 0 || t.argmax_variant != 0 || (g.HW & 3) != 0) return cudaSuccess;
    const size_t es = g.dtype == HEAD_F32 ? 4 : 2;
    if ((reinterpret_cast<uintptr_t>(head_v) & (4 * es - 1)) || (g.img_stride * es) % (4 * es) || (g.limb_off * es) % (4 * es)) return cudaSuccess;
    int C = t.argmax_cluster > 1 ? t.argmax_cluster : 0;
    if (!C) {
        if (n_mats * 2 > d->sms) return cudaSuccess;
        C = 8;
        while (C > 1 && n_mats * C > d->sms) C >>= 1;
    }
    while (C > 1 && g.S / C < 2) C >>= 1;
    if (C < 2 || C > 8 || (C & (C - 1))) return cudaSuccess;
    const int CV = g.HW / 4;
    if (CV > 1024) return cudaSuccess;
    const int rows = (g.S + C - 1) / C;
    int G = 512 / CV;                                  // CTAs of at most 512 threads: two fit on an SM, so that 17 clusters of 8
    if (G < 1) G = 1;                                  // (native shape, one image) are resident at once — with 1024-thread CTAs
                                                       // the last cluster found no free GPC and ran as a second wave (16.7 -> 20.8 us)
    if (G > (rows + 1) / 2) G = (rows + 1) / 2;        // at least two rows per group
    if (G < 1) G = 1;
    while (G > 1 && CV * G > 1024) --G;
    const int threads = std::max(64, ((CV * G + 31) / 32) * 32);
    size_t smem = (size_t)G * g.HW * sizeof(Partial);
    // ring of bulk copies when rows are whole 16-byte units (always so for fp32: HW % 4 == 0): 4 stages of ~16 KB, so
    // that two CTAs still share an SM (see the note on G above)
    int ring_rows = 0;
    const size_t row_bytes = (size_t)g.HW * es;
    if (t.argmax_cluster_ring && row_bytes % 16 == 0 && (reinterpret_cast<uintptr_t>(head_v) & 15) == 0 &&
        (g.img_stride * es) % 16 == 0 && (g.limb_off * es) % 16 == 0 && row_bytes <= 32 * 1024) {
        ring_rows = (int)std::max<size_t>(1, (16 * 1024) / row_bytes);
        ring_rows = std::min(ring_rows, std::max(1, (rows + 3) / 4));
        smem = ((smem + 16 * sizeof(uint64_t) + 127) & ~(size_t)127) + (size_t)4 * ring_rows * row_bytes;
    }
    if (smem > (size_t)d->smem_optin) return cudaSuccess;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(n_mats * C));
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 2 : 1;
    cudaError_t e = cudaSuccess;
    PPN_DISPATCH_HEAD(g.dtype, {
        if ((e = ensure_smem(limb_argmax_cluster_kernel<T>, smem, &d->cluster[g.dtype])) != cudaSuccess) return e;
        e = cudaLaunchKernelEx(&cfg, limb_argmax_cluster_kernel<T>, static_cast<const T*>(head_v), amax, g, CV, G, pdl_bits, zero2, ring_rows);
    });
    if (e == cudaSuccess) *done = true;
    return e;
}

cudaError_t launch_limb_argmax(const void* head_v, uint16_t* amax, const Geom& g, const Tuning& t, cudaStream_t st,
                               bool pdl, bool* pdl_used, int pdl_bits, int32_t* zero2, bool* zeroed) {
    if (pdl_used) *pdl_used = false;
    if (zeroed) *zeroed = false;
    if (pdl_bits < 0) pdl_bits = pdl ? (PDL_TRIGGER | PDL_WAIT_END) : 0;
    DeviceInfo* d = nullptr;
    cudaError_t e = device_info(&d);
    if (e != cudaSuccess) return e;
    const int n_mats = g.B * g.E;
    if (n_mats == 0) return cudaSuccess;
    {
        bool done = false;
        e = try_launch_argmax_cluster(head_v, amax, g, t, st, pdl, pdl_bits, d, zero2, &done);
        if (e != cudaSuccess) return e;
        if (done) {
            if (pdl_used) *pdl_used = pdl;
            if (zeroed) *zeroed = zero2 != nullptr;
            return cudaSuccess;
        }
    }
    if (g.dtype == HEAD_F16)
        return launch_limb_argmax16(static_cast<const __half*>(head_v), amax, g, t, st, pdl, pdl_used, pdl_bits, d, &d->tma16[0], zero2, zeroed);
    if (g.dtype == HEAD_BF16)
        return launch_limb_argmax16(static_cast<const __nv_bfloat16*>(head_v), amax, g, t, st, pdl, pdl_used, pdl_bits, d, &d->tma16[1], zero2, zeroed);
    if (g.dtype != HEAD_F32) return cudaErrorInvalidValue;
    const float* head = static_cast<const float*>(head_v);
    ArgmaxPlan p;
    const bool vec_ok = plan_argmax(g, t, d->sms, &p) && ((reinterpret_cast<uintptr_t>(head) & 15) == 0);
    if (vec_ok && t.argmax_variant == 0) {
        // shrink the ring until it fits the opt-in shared memory (split between resident CTAs)
        size_t budget = (size_t)d->smem_optin / p.ctas_per_sm - (p.ctas_per_sm > 1 ? 1024 : 0);
        {   // honour the per-call cap if a ring of at least two stages fits under it
            const size_t two = p.smem_bytes - (size_t)(p.stages - 2) * (p.stage_bytes + 2 * sizeof(uint64_t) + sizeof(int));
            if (t.argmax_smem_cap > 0 && (size_t)t.argmax_smem_cap < budget && (p.stages < 2 || two <= (size_t)t.argmax_smem_cap))
                budget = (size_t)t.argmax_smem_cap;
        }
        while (p.smem_bytes > budget && p.stages > 2) {
            --p.stages;
            p.smem_bytes -= p.stage_bytes + 2 * sizeof(uint64_t) + sizeof(int);
        }
        if (p.smem_bytes <= budget) {
            int* ticket = nullptr;
            if (t.argmax_dynamic && (e = ticket_for(d, st, &ticket)) != cudaSuccess) return e;
            int grid = d->sms * p.ctas_per_sm;
            if (p.split_mats) {
                const int n_items = item_count(p, n_mats);
                if (grid > n_items) grid = n_items;
                if ((e = ensure_smem(limb_argmax_tma_multi_kernel, p.smem_bytes, &d->tma_multi)) != cudaSuccess) return e;
                e = launch_kernel(limb_argmax_tma_multi_kernel, dim3(grid), dim3(p.threads_padded + 32), p.smem_bytes, st, pdl,
                                  head, amax, g, p, pdl_bits, ticket, zero2);
            } else {
                if (grid > n_mats) grid = n_mats;
                if ((e = ensure_smem(limb_argmax_tma_kernel, p.smem_bytes, &d->tma)) != cudaSuccess) return e;
                e = launch_kernel(limb_argmax_tma_kernel, dim3(grid), dim3(p.threads_padded + 32), p.smem_bytes, st, pdl,
                                  head, amax, g, p, pdl_bits, ticket, zero2);
            }
            if (pdl_used) *pdl_used = pdl;
            if (zeroed) *zeroed = zero2 != nullptr;
            return e;
        }
    }
    if (vec_ok) {
        if (p.split_mats) {                     // the direct-load kernel always splits rows
            Tuning rows_mode = t;
            rows_mode.argmax_split = 0;
            plan_argmax(g, rows_mode, d->sms, &p);
        }
        const size_t smem = (size_t)p.G * g.HW * sizeof(Partial);
        if ((e = ensure_smem(limb_argmax_ldg_kernel, smem, &d->ldg)) != cudaSuccess) return e;
        limb_argmax_ldg_kernel<<<n_mats, p.threads_padded, smem, st>>>(head, amax, g, p);
        return cudaGetLastError();
    }
    dim3 grid(n_mats, (g.HW + 255) / 256);
    limb_argmax_generic_kernel<float><<<grid, 256, 0, st>>>(head, amax, g);
    return cudaGetLastError();
}

cudaError_t launch_decode_candidates(const void* head, const Geom& g, int n_parts, float thr, int32_t* cand_cell,
                                     float* cand_score, float* cand_box, int32_t* cand_count, cudaStream_t st) {
    if (g.B == 0 || n_parts == 0) return cudaSuccess;
    dim3 grid(g.B, n_parts);
    PPN_DISPATCH_HEAD(g.dtype, decode_candidates_kernel<T><<<grid, 256, 0, st>>>(
        static_cast<const T*>(head), g, n_parts, thr, cand_cell, cand_score, reinterpret_cast<float4*>(cand_box), cand_count));
    return cudaGetLastError();
}

cudaError_t launch_restore_xy(const float* x, const float* y, float* rx, float* ry, size_t n, int H, int W,
                              float gridW, float gridH, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    restore_xy_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, y, rx, ry, n, H * W, W, gridW, gridH);
    return cudaGetLastError();
}

cudaError_t launch_restore_size(const float* w, const float* h, float* rw, float* rh, size_t n, float inW, float inH,
                                cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    restore_size_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(w, h, rw, rh, n, inW, inH);
    return cudaGetLastError();
}

size_t nms_smem_bytes(int stride) { return nms_bytes_per_list(stride); }

// benchmark knob "nms.blockwise" (ppn_tune): process-wide, read at launch time
static std::atomic<int> g_nms_blockwise{0};
void set_nms_blockwise(int on) { g_nms_blockwise.store(on != 0); }
int get_nms_blockwise() { return g_nms_blockwise.load(); }

cudaError_t launch_nms(const float* box, const float* score, const int32_t* count, int n_problems, int stride,
                       float thr, int limit, int32_t* keep_idx, int32_t* keep_count, cudaStream_t st) {
    if (n_problems == 0) return cudaSuccess;
    DeviceInfo* d = nullptr;
    cudaError_t e = device_info(&d);
    if (e != cudaSuccess) return e;
    const size_t smem = nms_smem_bytes(stride);
    if (stride <= 1024 && smem <= (size_t)d->smem_optin) {
        if ((e = ensure_smem(nms_smem_kernel, smem, &d->nms)) != cudaSuccess) return e;
        nms_smem_kernel<<<n_problems, stride <= 256 ? 256 : 512, smem, st>>>(reinterpret_cast<const float4*>(box), score, count,
                                                                             stride, thr, limit, keep_idx, keep_count,
                                                                             g_nms_blockwise.load());
        return cudaGetLastError();
    }
    nms_global_kernel<<<n_problems, 1024, 0, st>>>(reinterpret_cast<const float4*>(box), score, count, stride, thr,
                                                   limit, keep_idx, keep_count);
    return cudaGetLastError();
}

cudaError_t launch_part_centres(const int32_t* count, const int32_t* cell, const float* box, int B, int R, int K,
                                float* centre, cudaStream_t st) {
    const size_t n = (size_t)B * R * K;
    if (n == 0) return cudaSuccess;
    part_centres_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(count, cell, reinterpret_cast<const float4*>(box), n, R, K,
                                                                     reinterpret_cast<float2*>(centre));
    return cudaGetLastError();
}

cudaError_t launch_skeleton(const int32_t* count, const int32_t* cell, const float* box, int B, int R, int K, int E,
                            const int32_t* edges, int32_t* rect, float* keypoint, float* segment, cudaStream_t st) {
    const size_t n = (size_t)B * R * (1 + K + E);
    if (n == 0) return cudaSuccess;
    EdgePairs ep;
    for (int e = 0; e < E; ++e) { ep.src[e] = (uint8_t)edges[2 * e]; ep.dst[e] = (uint8_t)edges[2 * e + 1]; }
    skeleton_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(count, cell, reinterpret_cast<const float4*>(box), n, R, K, E, ep,
                                                                 reinterpret_cast<int4*>(rect), reinterpret_cast<float2*>(keypoint),
                                                                 reinterpret_cast<float4*>(segment));
    return cudaGetLastError();
}

cudaError_t launch_pack_humans(const int32_t* count, const int32_t* cell, const float* score, const float* box, int B, int R,
                               int K, int cap, int32_t* header, uint32_t* e_idcell, float* e_score, float* e_box,
                               cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    pack_count_kernel<<<B, 256, 0, st>>>(count, cell, R, K, header, B);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const size_t smem = (size_t)(R + 1) * sizeof(int);
    DeviceInfo* d = nullptr;
    if ((e = device_info(&d)) != cudaSuccess) return e;
    if (smem > (size_t)d->smem_optin) return cudaErrorInvalidConfiguration;
    static size_t have[64] = {};
    int dev = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if (smem > 48 * 1024 && (e = ensure_smem(pack_entries_kernel, smem, &have[dev & 63])) != cudaSuccess) return e;
    pack_entries_kernel<<<B, 256, smem, st>>>(count, cell, score, reinterpret_cast<const float4*>(box),
                                                                        B, R, K, cap, header, e_idcell, e_score,
                                                                        reinterpret_cast<float4*>(e_box));
    return cudaGetLastError();
}

size_t decode_nms_smem_bytes(const Geom& g) {
    return (size_t)g.HW * sizeof(float4) + (size_t)((g.HW + 3) & ~3) * sizeof(int32_t) + nms_smem_bytes(g.HW);
}

cudaError_t launch_decode_nms(const void* head, const Geom& g, int n_parts, float det_thr, float nms_thr,
                              int32_t* keep_cell, int32_t* keep_count, cudaStream_t st, bool pdl_attr, int pdl_bits,
                              int ctas_per_sm, int threads_pref) {
    if (g.B == 0 || n_parts == 0) return cudaSuccess;
    DeviceInfo* d = nullptr;
    cudaError_t e = device_info(&d);
    if (e != cudaSuccess) return e;
    const size_t smem = decode_nms_smem_bytes(g);
    if (smem > (size_t)d->smem_optin) return cudaErrorInvalidConfiguration;
    // persistent: at most ctas_per_sm CTAs per SM, each striding over the (image, part) lists (0: one CTA per list)
    const long long lists = (long long)g.B * n_parts;
    dim3 grid((unsigned)(ctas_per_sm > 0 ? std::min<long long>(lists, (long long)d->sms * ctas_per_sm) : lists));
    PPN_DISPATCH_HEAD(g.dtype, {
        if ((e = ensure_smem(decode_nms_kernel<T>, smem, &d->decode_nms[g.dtype])) != cudaSuccess) return e;
        const int threads = threads_pref > 0 ? std::min(512, std::max(64, (threads_pref + 31) & ~31)) : (g.HW <= 256 ? 256 : 512);
        return launch_kernel(decode_nms_kernel<T>, grid, dim3(threads), smem, st, pdl_attr,
                             static_cast<const T*>(head), g, n_parts, det_thr, nms_thr, keep_cell, keep_count,
                             pdl_bits | (g_nms_blockwise.load() ? NMS_BLOCKWISE : 0));
    });
    return cudaErrorInvalidValue;
}

static size_t head_elem_bytes(int dtype) { return dtype == HEAD_F32 ? 4 : 2; }

// parts whose x / y / w / h planes the tree parse brings into shared memory at a time for crowded images: as many as
// fit in 24 KB, and only where that means a handful of passes over the K parts (small grids — where crowds are dense)
static int tree_parse_xywh_parts(const Geom& g, int n_groups) {
    if (n_groups >= 6) return 0;
    const size_t per_part = (size_t)4 * g.HW * head_elem_bytes(g.dtype);
    int P = (int)((24 * 1024) / per_part);
    if (P > g.K) P = g.K;
    return (P >= 1 && (g.K + P - 1) / P <= 4) ? P : 0;
}

static size_t tree_parse_smem_base(const Geom& g, int n_groups) {
    return ((((size_t)n_groups * g.K * g.HW * head_elem_bytes(g.dtype)) + 15) & ~(size_t)15) +
           ((((size_t)g.E * g.HW + 7) & ~(size_t)7)) * sizeof(uint16_t) +
           (size_t)2 * g.HW * sizeof(int32_t) + (g.S <= kMaxDyxTable ? (size_t)g.S * sizeof(int32_t) : 0) +
           ((((size_t)g.HW * g.K * sizeof(int16_t)) + 15) & ~(size_t)15);
}

size_t tree_parse_smem_bytes(const Geom& g, int n_groups) {
    const int P = tree_parse_xywh_parts(g, n_groups);
    return tree_parse_smem_base(g, n_groups) + (P ? 16 + (size_t)P * 4 * g.HW * head_elem_bytes(g.dtype) : 0);   // + alignment slack
}

// How much of the decode block the tree parse stages in shared memory (stage_all_pref: -1 auto, 0 none,
// 1 resp+conf, 2 all six groups).  Auto: all six when that keeps the CTA under 32 KB (tiny
// grids), resp+conf when under 64 KB (cfg2: 25 KB, cfg3: 57 KB), nothing otherwise — a light CTA lets every
// image be resident at once, several of them UNDER the arg-max ring, and under the next call's
// kernels (measured: at 24x24 the 107 KB staged CTA shut both overlaps out).
static int tree_parse_groups(const Geom& g, int stage_all_pref, int smem_optin) {
    int n_groups;
    if (stage_all_pref < 0)
        n_groups = tree_parse_smem_base(g, 6) <= 32 * 1024 ? 6 : (tree_parse_smem_base(g, 2) <= 64 * 1024 ? 2 : 0);
    else
        n_groups = stage_all_pref >= 2 ? 6 : (stage_all_pref == 1 ? 2 : 0);
    while (n_groups > 0 && tree_parse_smem_bytes(g, n_groups) > (size_t)smem_optin) n_groups = n_groups == 6 ? 2 : 0;
    return n_groups;
}

// Shared memory left for the arg-max ring on an SM when `k12_ctas` decode+NMS CTAs and one tree-parse CTA are to be
// resident beside it (the persistent three-kernel chain); 0 when they would leave less than a two-stage ring.
size_t chain3_ring_cap(const Geom& g, int stage_all_pref, int k12_ctas) {
    DeviceInfo* d = nullptr;
    if (device_info(&d) != cudaSuccess) return 0;
    const size_t sm_bytes = (size_t)d->smem_optin + 1024;
    const size_t others = (size_t)k12_ctas * (decode_nms_smem_bytes(g) + 1024) +
                          tree_parse_smem_bytes(g, tree_parse_groups(g, stage_all_pref, d->smem_optin)) + 1024;
    if (others + 1024 + 64 * 1024 > sm_bytes) return 0;
    return sm_bytes - others - 1024;
}

cudaError_t launch_tree_parse(const void* head, const Geom& g, const ChainTable& ch, float thr, int min_kp, int n_parts,
                              const uint16_t* amax, const int32_t* cand_cell, const int32_t* keep_idx,
                              const int32_t* keep_count, int32_t* h_count, int32_t* h_root, int32_t* h_cell,
                              float* h_score, float* h_box, int R, cudaStream_t st, bool pdl_attr, int pdl_bits,
                              int stage_all_pref, int threads_pref, int chain_mode, int ctas_per_sm) {
    if (g.B == 0) return cudaSuccess;
    DeviceInfo* d = nullptr;
    cudaError_t e = device_info(&d);
    if (e != cudaSuccess) return e;
    const int n_groups = tree_parse_groups(g, stage_all_pref, d->smem_optin);
    const size_t smem = tree_parse_smem_bytes(g, n_groups);
    // one thread per (chain, root) in the walk and per (human, part) pair in the write-out
    int threads = threads_pref > 0 ? threads_pref : ((g.HW <= 144 || n_groups == 0) ? 256 : 512);
    threads = ((threads < 64 ? 64 : (threads > 1024 ? 1024 : threads)) + 31) & ~31;
    if (smem > (size_t)d->smem_optin) return cudaErrorInvalidConfiguration;
    // bulk copies need 16-byte sizes and sources: the staged planes are es*n*K*HW bytes at image
    // offset es*C*HW*b (es = element size), the arg-max map 2*E*HW bytes at offset 2*E*HW*b
    const size_t es = head_elem_bytes(g.dtype);
    const bool tma_ok = ((size_t)g.K * g.HW * 2 * es) % 16 == 0 && (g.img_stride * es) % 16 == 0 &&
                        ((size_t)g.E * g.HW * 2) % 16 == 0 && (reinterpret_cast<uintptr_t>(head) & 15) == 0 &&
                        (reinterpret_cast<uintptr_t>(amax) & 15) == 0;
    // persistent: at most ctas_per_sm CTAs per SM, each striding over the images (0: one CTA per image)
    const dim3 grid((unsigned)(ctas_per_sm > 0 ? std::min<long long>(g.B, (long long)d->sms * ctas_per_sm) : g.B));
    // chain_mode 0: pdl_bits as given; 1: a publishing link of the call chain that triggers after its wait;
    //            2: overlapped calls — guard on the previous call's publication, trigger at the very top
    StreamSlot* slot = nullptr;
    int* words = nullptr;
    int bits = pdl_bits, seq = 0;
    if (chain_mode > 0) {
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if ((e = cudaStreamIsCapturing(st, &cap)) != cudaSuccess) return e;
        if (cap == cudaStreamCaptureStatusNone && (e = slot_for(d, st, &slot, &words)) != cudaSuccess) return e;
        if (slot) { bits |= FUSED_PUBLISH; seq = slot->published; }
        if (pdl_attr && chain_mode == 2 && slot) bits = (bits & ~PDL_TRIGGER) | FUSED_GUARD | FUSED_TRIGGER_EARLY;
    }
    int* sync = words ? words + 4 : nullptr;
    PPN_DISPATCH_HEAD(g.dtype, {
        if (n_groups) {
            if ((e = ensure_smem(tree_parse_kernel<true, T>, smem, &d->tree[g.dtype])) != cudaSuccess) return e;
            e = launch_kernel(tree_parse_kernel<true, T>, grid, dim3(threads), smem, st, pdl_attr, static_cast<const T*>(head),
                              g, ch, thr, min_kp, n_parts, amax, cand_cell, keep_idx, keep_count, h_count, h_root, h_cell,
                              h_score, reinterpret_cast<float4*>(h_box), R, tma_ok ? 1 : 0, n_groups, bits, sync, seq,
                              tree_parse_xywh_parts(g, n_groups));
        } else {
            if ((e = ensure_smem(tree_parse_kernel<false, T>, smem, &d->tree_light[g.dtype])) != cudaSuccess) return e;
            e = launch_kernel(tree_parse_kernel<false, T>, grid, dim3(threads), smem, st, pdl_attr, static_cast<const T*>(head),
                              g, ch, thr, min_kp, n_parts, amax, cand_cell, keep_idx, keep_count, h_count, h_root, h_cell,
                              h_score, reinterpret_cast<float4*>(h_box), R, tma_ok ? 1 : 0, n_groups, bits, sync, seq,
                              tree_parse_xywh_parts(g, n_groups));
        }
    });
    if (e == cudaSuccess && slot) {
        std::lock_guard<std::mutex> lock(g_ticket_mu);
        slot->published = seq + 1;
        slot->fast_open = true;
    }
    return e;
}

// ---- fused decode + NMS + tree parse --------------------------------------------------------------
// Staging delta (K*HW floats) makes every walk step and score a shared-memory read; it costs shared
// memory, i.e. parse CTAs per SM beside the arg-max ring.  stage_pref: -1 auto, 0 never, >= 1 whenever
// it fits at all.
//
// The overlapped chain needs EVERY parse CTA of a launch resident beside one arg-max CTA per SM
// (threads, registers, shared memory with a ring of at least three 32 KB stages).  A batch too large
// for that is cut into equal sub-batches that do fit, each with its own arg-max + parse launch pair:
// sub-batch j+1's arg-max then streams while sub-batch j is parsed, exactly like consecutive calls.
static int fused_ctas_per_sm(const Geom& g, const Tuning& t, int smem_optin, size_t smem) {
    const int t124 = g.HW <= 256 ? 256 : 512;
    // the arg-max CTA: consumer threads + producer warp, 56 registers per thread (ptxas)
    const int t3 = ((g.dtype == HEAD_F32 ? t.argmax_threads : t.argmax16_threads) + 31) / 32 * 32 + 32;
    const size_t sm_bytes = (size_t)smem_optin + 1024;             // per SM: the opt-in maximum + one CTA's reserve
    const size_t min_ring = 3 * 32 * 1024 + 1024;
    if (smem > (size_t)smem_optin || sm_bytes < min_ring + 1024) return 0;
    long long n = (2048 - t3) / t124;
    n = std::min<long long>(n, (65536 - (long long)t3 * 56) / ((long long)t124 * 40));
    n = std::min<long long>(n, (long long)((sm_bytes - min_ring - 1024) / (smem + 1024)));
    return n < 0 ? 0 : (int)n;
}

static bool fused_split_plan(const Geom& g, const Tuning& t, DeviceInfo* d, int stage_pref, FusedSplit* out) {
    if (g.HW > 1024 || g.B < 1) return false;                      // the NMS bit matrix is built for <= 1024 boxes
    const size_t with = fused_layout(g, true).total, without = fused_layout(g, false).total;
    const int cap_with = stage_pref == 0 ? 0 : fused_ctas_per_sm(g, t, d->smem_optin, with) * d->sms;
    const int cap_without = stage_pref > 0 ? 0 : fused_ctas_per_sm(g, t, d->smem_optin, without) * d->sms;
    const int n_with = cap_with > 0 ? (g.B + cap_with - 1) / cap_with : 0;
    const int n_without = cap_without > 0 ? (g.B + cap_without - 1) / cap_without : 0;
    if (!n_with && !n_without) return false;
    // fewer launch pairs win; at equal count staged delta (shorter walk chain) if the CTA stays under 48 KB
    bool staged = n_with && (!n_without || n_with < n_without || (n_with == n_without && (stage_pref > 0 || with <= 48 * 1024)));
    out->staged = staged;
    out->smem = staged ? with : without;
    out->n_sub = staged ? n_with : n_without;
    out->sub_B = (g.B + out->n_sub - 1) / out->n_sub;
    const int per_sm = (out->sub_B + d->sms - 1) / d->sms;
    out->ring_cap = (size_t)d->smem_optin + 1024 - (size_t)per_sm * (out->smem + 1024) - 1024;
    return true;
}

// Fallback shape when nothing fits beside a ring: one CTA per image, whatever staging fits at all.
static bool fused_plan(const Geom& g, int smem_optin, int stage_pref, bool* staged, size_t* smem) {
    if (g.HW > 1024) return false;
    const size_t with = fused_layout(g, true).total, without = fused_layout(g, false).total;
    bool st = stage_pref < 0 ? with <= 48 * 1024 : (stage_pref > 0 && with <= (size_t)smem_optin);
    if (!st && without > (size_t)smem_optin) return false;
    *staged = st;
    *smem = st ? with : without;
    return true;
}

bool parse_fused_supported(const Geom& g, int stage_pref) {
    DeviceInfo* d = nullptr;
    if (device_info(&d) != cudaSuccess) return false;
    bool staged;
    size_t smem;
    return fused_plan(g, d->smem_optin, stage_pref, &staged, &smem);
}

bool parse_fused_split(const Geom& g, int stage_pref, const Tuning& t, FusedSplit* out) {
    DeviceInfo* d = nullptr;
    if (device_info(&d) != cudaSuccess) return false;
    return fused_split_plan(g, t, d, stage_pref, out);
}

size_t parse_fused_smem_bytes(const Geom& g, int stage_pref) {
    DeviceInfo* d = nullptr;
    bool staged;
    size_t smem = 0;
    if (device_info(&d) != cudaSuccess || !fused_plan(g, d->smem_optin, stage_pref, &staged, &smem)) return 0;
    return smem;
}

cudaError_t launch_parse_fused(const void* head, const Geom& g, const ChainTable& ch, float det_thr, float nms_thr, int min_kp,
                               const uint16_t* amax, int32_t* h_count, int32_t* h_root, int32_t* h_cell, float* h_score,
                               float* h_box, int R, cudaStream_t st, bool pdl_attr, int chain_mode, int stage_pref,
                               int staged_forced, const DenseTarget* dense_to, bool wait_top) {
    if (g.B == 0) return cudaSuccess;
    DeviceInfo* d = nullptr;
    cudaError_t e = device_info(&d);
    if (e != cudaSuccess) return e;
    bool staged;
    size_t smem;
    if (!fused_plan(g, d->smem_optin, stage_pref, &staged, &smem)) return cudaErrorInvalidConfiguration;
    if (staged_forced >= 0) {                                      // the caller planned the staging (sub-batches)
        staged = staged_forced != 0;
        smem = fused_layout(g, staged).total;
        if (smem > (size_t)d->smem_optin) return cudaErrorInvalidConfiguration;
    }
    DenseOut dense = {nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, 0, 0};
    if (dense_to) {
        if (g.K > 32) return cudaErrorInvalidConfiguration;          // present-part masks are 32 bits
        dense = DenseOut{dense_to->header, dense_to->rheader, dense_to->idcell, dense_to->score, reinterpret_cast<float4*>(dense_to->box),
                         dense_to->cap, dense_to->skip_slots, dense_to->B_total, dense_to->b0};
    }
    // chain_mode 0: plain launch; 1: programmatic dependent that triggers after its wait;
    //            2: overlapped calls — guard, early trigger (see the kernel's header comment)
    StreamSlot* slot = nullptr;
    int* words = nullptr;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if ((e = cudaStreamIsCapturing(st, &cap)) != cudaSuccess) return e;
    if (cap == cudaStreamCaptureStatusNone && (e = slot_for(d, st, &slot, &words)) != cudaSuccess) return e;
    int bits = 0;
    if (pdl_attr) bits |= PDL_WAIT_START;
    if (pdl_attr && wait_top) bits |= FUSED_WAIT_TOP;
    int seq = 0;
    if (slot) { bits |= FUSED_PUBLISH; seq = slot->published; }
    if (pdl_attr && chain_mode == 2 && slot) bits |= FUSED_GUARD | FUSED_TRIGGER_EARLY;
    else if (pdl_attr) bits |= PDL_TRIGGER;
    if (g_nms_blockwise.load()) bits |= NMS_BLOCKWISE;
    const int threads = g.HW <= 256 ? 256 : 512;
    int* sync = words ? words + 4 : nullptr;
    PPN_DISPATCH_HEAD(g.dtype, {
        if (staged) {
            if ((e = ensure_smem(parse_fused_kernel<true, T>, smem, &d->fused[1][g.dtype])) != cudaSuccess) return e;
            e = launch_kernel(parse_fused_kernel<true, T>, dim3(g.B), dim3(threads), smem, st, pdl_attr, static_cast<const T*>(head), g, ch,
                              det_thr, nms_thr, min_kp, amax, h_count, h_root, h_cell, h_score, reinterpret_cast<float4*>(h_box), R,
                              bits, sync, seq, dense);
        } else {
            if ((e = ensure_smem(parse_fused_kernel<false, T>, smem, &d->fused[0][g.dtype])) != cudaSuccess) return e;
            e = launch_kernel(parse_fused_kernel<false, T>, dim3(g.B), dim3(threads), smem, st, pdl_attr, static_cast<const T*>(head), g, ch,
                              det_thr, nms_thr, min_kp, amax, h_count, h_root, h_cell, h_score, reinterpret_cast<float4*>(h_box), R,
                              bits, sync, seq, dense);
        }
    });
    if (e == cudaSuccess && slot) {
        std::lock_guard<std::mutex> lock(g_ticket_mu);
        slot->published = seq + 1;
        slot->fast_open = true;
    }
    return e;
}

// May the next arg-max launch on `st` start beside the stream's previous parse?  Only when that was a
// publishing fused parse (or nothing of ours): any other whole-path launch calls chain_break().
bool chain_clean(cudaStream_t st) {
    DeviceInfo* d = nullptr;
    if (device_info(&d) != cudaSuccess) return false;
    std::lock_guard<std::mutex> lock(g_ticket_mu);
    for (int i = 0; i < d->slots_used; ++i)
        if (d->slot[i].stream == st) return d->slot[i].fast_open;
    return false;
}

void chain_break(cudaStream_t st) {
    DeviceInfo* d = nullptr;
    if (device_info(&d) != cudaSuccess) return;
    std::lock_guard<std::mutex> lock(g_ticket_mu);
    for (int i = 0; i < d->slots_used; ++i)
        if (d->slot[i].stream == st) d->slot[i].fast_open = false;
}

}  // namespace ppn
