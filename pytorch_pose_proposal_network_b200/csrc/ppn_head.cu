// Fused network head: the final 1x1 convolution (model.py:85 `conv3 = Conv2d(512, lastsize, 1)`), the
// sigmoid (model.py:133-136) and the limb-window arg-max of the parser (datatest.py:100,113) in ONE
// kernel, so that the fp32 head tensor [B, 6K + S*E, H, W] — 17.5 MB per image at the reference's shape,
// 98.6 % of it limb values whose only use is one arg-max per window — is never written to HBM nor
// read back.  What leaves the kernel is the 6K decode planes (sigmoid applied) and the uint16 arg-max
// map; the fused decode + NMS + tree-parse kernel (ppn_kernels.cu, K124) consumes both.
//
// The 1x1 convolution is a GEMM per image, D[cell, c] = sum_k X[b, k, cell] * W[c, k] (+ bias[c]):
//   A = X_b^T  [M = cells,    K = Cin]   "MN-major" in memory (cells contiguous: NCHW activations)
//   B = W      [N = channels, K = Cin]   K-major
// computed on the 5th-generation tensor cores: tcgen05.mma kind::tf32 (fp32 operands read from shared
// memory, fp32 accumulation — the precision class of the reference's own cuDNN convolution, which
// PyTorch runs in TF32 by default), 128 x 256 accumulator tiles in tensor memory (TMEM), operands
// brought in by TMA (cp.async.bulk.tensor, 128-byte swizzle; 32-byte swizzle atoms for the MN-major
// activations) through a 4-stage mbarrier ring.
// Cells are the M dimension on purpose: an accumulator row (TMEM lane) then belongs to ONE cell and
// the epilogue thread that owns the lane scans the channels in order, keeping numpy's running
// (max, first index) per limb window in registers — the same per-thread rule as the streaming
// arg-max kernel, no cross-lane reduction.  The accumulator is double-buffered (2 x 256 TMEM columns):
// the epilogue of channel tile n runs under the MMAs of tile n + 1.
//
// Warp roles (192 or 448 threads, one CTA per SM, persistent over M tiles):
//   warp 0      TMA producer (one lane)
//   warp 1      TMEM allocation, MMA issue (one lane), TMEM release
//   warps 2-5 (or 2-13: three per TMEM lane quadrant, for short limb windows)
//               epilogue: TMEM -> registers (tcgen05.ld 32x32b), bias, sigmoid / running arg-max, stores
//
// M tiles are built from "cell groups" of 32 cells of one image (a 128-byte swizzle row): a tile is 4
// consecutive groups of the flattened (image, group) list, each fetched by its own TMA box from the
// 3-D view [B][Cin][HW] with zero fill past HW — so a 12x12 grid (144 = 4.5 groups) wastes 11 % of
// the rows, not 44 %, and every epilogue warp (one group) works on a single image.
//
// Two operand paths (HeadOperand): TF32 on the fp32 NCHW activations read in place (above), and a 16-bit path
// (fp16 or bf16 operands, kind::f16, fp32 accumulation — what the reference's conv3 computes under its apex AMP
// training setup, main.py:282-289): a pre-pass packs activations and weights K-major in 16 bits (or the caller hands
// in channels_last 16-bit activations), the A tile of a block of 128 cells stays resident in shared memory for all
// channel tiles and only the weights stream.  See head_gemm16_argmax_kernel.
//
// Exactness.  The parser's contract is "bit-exact on sigmoid(logits)".  sigmoid is monotone but not
// injective in fp32 (neighbouring logits often share a sigmoid value), so an arg-max over logits can
// differ from numpy's first-maximum over the sigmoid values.  The running rule therefore decides on
// sigmoid values — but only a logit that exceeds the running maximum logit can change the answer, and
// of those only near-ties and the saturated tails need the two sigmoids evaluated (see the epilogue).
#include <cuda.h>          // CUtensorMap and enums only: the encoder is fetched with cudaGetDriverEntryPoint
#include <mutex>
#include <type_traits>

#include "ppn_kernels.h"

namespace ppn {

namespace {

constexpr int kBlockM = 128;                 // cells per accumulator tile (4 groups of 32)
constexpr int kBlockN = 256;                 // channels per accumulator tile
constexpr int kBlockK = 32;                  // fp32 elements per 128-byte swizzle row
constexpr int kUmmaK = 8;                    // tf32: 32 bytes of K per instruction
constexpr int kStages = 4;
constexpr int kGroupBytes = kBlockK * 128;   // one cell group of a stage: 32 k-rows x 128 B
constexpr int kABytes = 4 * kGroupBytes;     // 16 KB
constexpr int kBBytes = kBlockN * 128;       // 32 KB
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kTmemCols = 512;               // two 256-column accumulators

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {      // arrives on `bar` when every MMA issued so far has completed
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], one instruction of M x N x 32 bytes of K: kind 0 = tf32 (K = 8), 1 = f16 / bf16 (K = 16)
template <int kKind>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    if constexpr (kKind == 0)
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
            "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
    else
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
            "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// Shared-memory matrix descriptor (sm_100 format: version 1); offsets in bytes.  layout: 2 = 128-byte swizzle of
// 16-byte chunks (K-major operands), 1 = 128-byte swizzle of 32-byte chunks — the only layout the tensor core
// accepts for an MN-major operand of 32-bit elements (TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B); with the plain
// 128-byte swizzle the instruction is silently dropped (measured: all-zero accumulators).
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t leading_bytes, uint32_t stride_bytes, uint32_t layout) {
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)((leading_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((stride_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}
// 32 lanes x 8 consecutive columns of TMEM -> 8 registers per thread (thread = lane).  The load is asynchronous: the
// registers are defined only after tcgen05.wait::ld, which therefore takes them as read-write operands — the compiler
// then cannot move a use above the wait.  Issue the next group's load, process the current group, wait: the TMEM
// latency hides under the compares.  (Eight columns at a time in a ROLLED loop on purpose: the first version unrolled
// 32 columns with the sigmoid paths inlined — 7 752 SASS instructions, 26 % of all stall samples "no instruction":
// the four epilogue warps thrashed the instruction cache.)
__device__ __forceinline__ void tmem_ld8_issue(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld8_wait(uint32_t* r) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]) :: "memory");
}

// Waiting without eating the issue slots of the scheduler's working warps: between polls the thread sleeps.  (ncu, round 2:
// 30 % of the kernel's executed instructions were the try_wait / branch pairs of the producer, the MMA issuer and the
// epilogue warps that were ahead.)
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity, unsigned ns) {
    uint32_t done;
    for (;;) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) return;
        __nanosleep(ns);
    }
}

// When is a logit x above the running maximum m CERTAINLY a larger sigmoid value (as torch / numpy see them in fp32)?
// For x - m > kSureStep and |x| <= kSureRange: sigmoid' >= 2.46e-3 on [-6.001, 6], so the true sigmoids are >= 2.46e-6
// apart, while each evaluated sigmoid (expf <= 2 ulp, one add, one IEEE division) is within ~4 ulp <= 2.4e-7 of the
// truth: a factor 5 of margin; below zero the values shrink like e^x and so does their spacing — the relative gap
// stays >= 1e-3.  Everything else (near-ties, the saturated tails, NaN, +-inf) evaluates the two sigmoids.
// (Round 2 started with 0.01 / 8 — margin 7 — and 17 % of the 8-column groups had a lane inside the 0.01 band and went
// through the exact rescan; with 1e-3 it is ~2 %.)
constexpr float kSureStep = 1e-3f, kSureRange = 6.0f;

// sigmoid_f32 (ppn_device.cuh): torch.sigmoid's fp32 expression, libdevice expf, one add, one IEEE division

// Does a logit x that exceeds every logit so far beat the standing arg-max, whose logit is bx <= x?  numpy sees sigmoid
// values: only if sigmoid(x) > sigmoid(bx) (a tie keeps the earlier index), and never once a NaN stands.  Out of line:
// it runs a few times per limb window and must not be replicated into every column of the epilogue.
__device__ __noinline__ bool beats_in_sigmoid(float x, float bx) {
    const float sx = sigmoid_f32(x), sb = sigmoid_f32(bx);
    return !(sx <= sb) && sb == sb;
}

}  // namespace

struct HeadArgs {
    int32_t B, HW, Cin, C, n_dec, S, E;
    int32_t groups_per_img, n_groups, n_tiles, n_ntiles, n_kblocks;
    int32_t n_chunks, chunk_tiles, n_items;   // a work item = (cell tile, chunk of chunk_tiles consecutive channel tiles): small batches
                                              // spread one cell tile's channels over several CTAs (the key maxima merge them)
    int32_t acc_n, acc_stages;  // channels per accumulator tile and how many accumulators TMEM holds: 256 x 2 (TF32 path) or 128 x 4
    int32_t n_last;             // channels of the LAST channel tile, rounded up to 16: its MMAs and its weight box are that narrow
    int32_t n_rows;             // 16-bit path: B * HW rows of the packed activation matrix
    int32_t n_bstages;          // 16-bit path: stages of the weight ring
    int32_t bf16;               // 16-bit path: operands are bf16 (else fp16)
    int32_t dry;                // benchmarks only (tune key head.dry): the epilogue releases every accumulator unread
    uint32_t magic_S;           // ceil(2^32 / S): exact p / S for p < 2^22 (S <= 65535 and S * E channels)
    const float* bias;          // [C] or nullptr
    float* dec;                 // [B, n_dec, HW]   sigmoid of the 6K decode channels
    unsigned long long* keys;   // [B, E, HW]  running (sigmoid, ~position) maxima, zero before the kernel
    float* emit_logits;         // optional [B, C, HW]: conv output before the sigmoid (parity tests)
    float* emit_head;           // optional [B, C, HW]: the reference's head tensor, sigmoid(logits)
};

// work item -> cell tile and its range of channel tiles
__device__ __forceinline__ void head_item(const HeadArgs& a, int item, int& tile, int& nt0, int& nt1) {
    tile = item / a.n_chunks;
    nt0 = (item - tile * a.n_chunks) * a.chunk_tiles;
    nt1 = min(nt0 + a.chunk_tiles, a.n_ntiles);
}

// ------------------------------ epilogue (both operand paths) ------------------------------
// kSubs warps share each TMEM lane quadrant (32 accumulator rows = 32 cells).  Every channel tile's columns are cut
// into kSubs runs of whole 8-column groups and sub-warp s takes run s — the same share of every tile whatever the
// window size, so the sub-warps never wait for one another (no barrier between them: the bias comes through the
// read-only cache, the accumulator is released by per-warp arrivals).  A sub-warp's run crosses limb windows; each
// maximal stretch of one window inside a run is a PIECE: the thread scans it with numpy's running first-maximum rule
// and publishes (sigmoid of the winner, its window position) with ONE 64-bit atomic max on keys[b][ei][cell]:
//     key = sigmoid bits << 32 | ~position        (sigmoid in [0, 1]: bit order == value order; NaN -> 0xffffffff)
// so the largest sigmoid wins, equal sigmoids resolve to the smallest position, the first NaN beats everything —
// numpy.argmax over the whole window, whichever sub-warps, channel tiles or order the pieces came from.  The keys
// start at zero (memset) and head_amax_finalize_kernel turns them into the uint16 map.
// (Round-2 history: windows were owned by sub-warps and the bias was staged in shared memory behind a barrier per
// channel tile; ncu: 55 warp instructions per accumulator column — skip scans with two divisions per group, the
// per-column generic path at every window boundary — and 20 % of all samples at that barrier: 107 us per tile of
// 128 cells x 1311 channels, the same for TF32 and 16-bit operands.  The kernel was bound by its epilogue.)
// kDense: accumulator row r of tile t is row t * 128 + r of the flattened (image, cell) list (16-bit path: no padding);
// otherwise the tile is 4 cell groups of 32 cells of one image each (TF32 path).
__device__ __noinline__ void publish_piece(unsigned long long* slot, float bx, int idx, bool valid) {
    const float sb = sigmoid_f32(bx);
    const uint32_t hi = (sb != sb) ? 0xFFFFFFFFu : __float_as_uint(sb);
    if (valid) atomicMax(slot, ((unsigned long long)hi << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)idx));
}

// Decode channels of one group: the LOGITS go to dec (head_finalize_kernel applies the sigmoid in place — 6K sigmoids per
// cell inside the epilogue made the sub-warp that met them four times slower than its neighbours on that channel tile).
// Out of line, all address arithmetic inside: inlined, the compiler hoisted sixteen 64-bit address chains per group
// above the branch that almost never needs them (146 of 460 instructions per group, ncu round 2).
__device__ __noinline__ void decode_group(float* dec, int b, int c0, int cell, int HW, int n_dec,
                                          uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3, uint32_t r4, uint32_t r5, uint32_t r6, uint32_t r7,
                                          float b0, float b1, float b2, float b3, float b4, float b5, float b6, float b7,
                                          int j_lo, int j_hi, bool valid) {
    if (!valid) return;
    float* p = dec + ((size_t)b * n_dec + c0) * HW + cell;
    const uint32_t r[8] = {r0, r1, r2, r3, r4, r5, r6, r7};
    const float bs[8] = {b0, b1, b2, b3, b4, b5, b6, b7};
#pragma unroll
    for (int j = 0; j < 8; ++j)
        if (j >= j_lo && j < j_hi) p[(size_t)j * HW] = __fadd_rn(__uint_as_float(r[j]), bs[j]);
}
// a column of a call that also emits the logits and the head tensor (parity tests)
__device__ __noinline__ void emit_column(float* emit_logits, float* emit_head, int b, int c, int cell, int C, int HW, float x, bool valid) {
    if (!valid) return;
    const size_t at = ((size_t)b * C + c) * HW + cell;
    if (emit_logits) emit_logits[at] = x;
    if (emit_head) emit_head[at] = sigmoid_f32(x);
}

template <int kSubs, bool kDense>
__device__ __forceinline__ void head_epilogue(const HeadArgs& a, uint32_t tmem_base, uint64_t* tfull, uint64_t* tempty) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ew = warp & 3;                     // the TMEM lane quadrant this warp may read
    const int sub = (warp - 2) >> 2;             // which of the quadrant's warps
    const bool emit = a.emit_logits != nullptr || a.emit_head != nullptr;
    const bool bias_vec = a.bias != nullptr;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
        int tile, nt0, nt1;
        head_item(a, item, tile, nt0, nt1);
        int b, cell;
        bool valid;
        if constexpr (kDense) {
            const int r = tile * kBlockM + ew * 32 + lane;
            valid = r < a.n_rows;
            b = valid ? r / a.HW : 0;
            cell = valid ? r - b * a.HW : 0;
        } else {
            const int g = tile * 4 + ew;
            b = g / a.groups_per_img;
            cell = (g - b * a.groups_per_img) * 32 + lane;
            valid = g < a.n_groups && cell < a.HW;
            if (!valid) { b = 0; cell = 0; }
        }
        unsigned long long* const key0 = a.keys + (size_t)b * a.E * a.HW + cell;      // + ei * HW
        for (int nt = nt0; nt < nt1; ++nt) {
            const int c_tile = nt * a.acc_n;
            const int n_cols = min(a.acc_n, a.C - c_tile);            // > 0
            // this sub-warp's run of the tile: whole 8-column groups
            const int n8 = (n_cols + 7) >> 3, per = (n8 + kSubs - 1) / kSubs;
            const int r_lo = c_tile + min(sub * per, n8) * 8;
            const int r_hi = min(c_tile + min((sub + 1) * per, n8) * 8, c_tile + n_cols);
            mbar_wait_sleep(&tfull[acc], acc_phase, 40);
            tc_fence_after();
            if (r_lo < r_hi && !(a.dry & 1)) {
                const uint32_t t_row = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * a.acc_n) - (uint32_t)c_tile;
                // state of the piece being scanned: m = largest logit so far (+inf once a NaN has been taken: nothing may
                // follow the first NaN), idx = the arg-max so far (window position) and bx = the logit it stands on
                // (bx <= m: a larger logit whose sigmoid TIES with the standing one does not move the arg-max).  A piece
                // starts from (-inf, -inf, its first position): sigmoid(-inf) = 0 stands until something beats it.
                bool limb = false;
                int ei = 0, wbase = 0, seg_end = 0, idx = 0;
                float m = -INFINITY, bx = -INFINITY;
                auto begin = [&](int c) {                             // uniform
                    if (c < a.n_dec) { limb = false; seg_end = min(a.n_dec, r_hi); return; }
                    const int p = c - a.n_dec;                        // exact magic division, p < 2^22
                    ei = (int)(((unsigned long long)(unsigned)p * a.magic_S) >> 32);
                    const int aw = p - ei * a.S;
                    limb = true; wbase = c - aw; seg_end = min(wbase + a.S, r_hi);
                    m = -INFINITY; bx = -INFINITY; idx = aw;
                };
                // One limb column at window position aw, the exact rule.  A logit above the running maximum beats the standing
                // arg-max iff sigmoid(x) > sigmoid(bx) (numpy sees sigmoid values).  When it is a sure step (kSureStep,
                // kSureRange above) it certainly does, and m >= bx: three selects, no branch.  Only the rest branches out to
                // evaluate the two sigmoids.
                auto limb_column = [&](float x, int aw) {
                    const bool gt = !(x <= m);
                    const bool fast = gt && __fsub_rn(x, m) > kSureStep && fabsf(x) <= kSureRange;
                    idx = fast ? aw : idx;
                    bx = fast ? x : bx;
                    if (gt && !fast) {
                        if (beats_in_sigmoid(x, bx)) { idx = aw; bx = x; }
                        m = (x != x) ? INFINITY : x;
                    }
                    m = fast ? x : m;
                };
                auto load_group = [&](int c0, uint32_t* r, float* bs) {
                    tmem_ld8_issue(t_row + (uint32_t)c0, r);
                    if (bias_vec && c0 + 8 <= a.C) {
                        const float4 lo = __ldg(reinterpret_cast<const float4*>(a.bias + c0));
                        const float4 hi = __ldg(reinterpret_cast<const float4*>(a.bias + c0) + 1);
                        bs[0] = lo.x; bs[1] = lo.y; bs[2] = lo.z; bs[3] = lo.w; bs[4] = hi.x; bs[5] = hi.y; bs[6] = hi.z; bs[7] = hi.w;
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; ++j) bs[j] = (bias_vec && c0 + j < a.C) ? __ldg(a.bias + c0 + j) : -0.0f;   // x + (-0) == x
                    }
                };
                uint32_t cur[8];
                float bcur[8];
                // Speculative scan of columns [j_lo, j_hi) of the loaded group (uniform bounds; kFull: all eight, straight-line
                // code whose columns overlap in the pipeline).  No branch and no predicate on the chain through m: m' =
                // max(m, x); a column may move the arg-max only if it is FAST (a sure step, kSureStep / kSureRange: a certainly larger
                // sigmoid, see limb_column); a lane that meets anything else above its running maximum — a near-tie, a
                // saturated tail, NaN, +-inf — marks itself bad, restores the state the group started from and rescans its
                // columns with the exact rule.  (The branchy exact rule on every column cost ~120 cycles per column and warp:
                // each column's branch waits for the predicate chain of the column before it.)
                auto spec_scan = [&](auto full_tag, const uint32_t* cur, const float* bcur, int j_lo, int j_hi, int aw0) {
                    constexpr bool kFull = decltype(full_tag)::value;
                    if constexpr (kFull) {
                        // The hot loop's form, 7 instructions a column instead of 10: per column only the difference, "a sure
                        // step" (d > kSureStep), "nothing or a sure step" (else the group is rescanned), the LAST stepping
                        // column and the running maximum.  The range half of the sure-step rule moves to the group: steps
                        // only go up, so all stepping columns lie within [-kSureRange, kSureRange] iff the last one (= the
                        // final maximum) is <= kSureRange and the first one is >= -kSureRange, which holds when the maximum
                        // the group started from is (or, at the start of a piece, m = -inf, when column 0 is: it always
                        // steps).  A group that started from a finite maximum below -kSureRange and steps is simply rescanned.
                        // After a clean group with a step, bx = the final maximum (the last stepping column carries it; later
                        // columns are <= it) and idx = that column; arg-max and bx are not touched inside the loop.
                        const float m0 = m;
                        bool good = true;
                        int js = -1;
                        float x0 = 0.0f;
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float x = __fadd_rn(__uint_as_float(cur[j]), bcur[j]);
                            if (j == 0) x0 = x;
                            const float d = __fsub_rn(x, m);
                            const bool step = d > kSureStep;
                            good = good && (d <= 0.0f || step);          // NaN differences fail both
                            js = step ? j : js;
                            m = fmaxf(m, x);
                        }
                        const bool any = js >= 0;
                        const bool in_range = m <= kSureRange && (m0 >= -kSureRange || (m0 == -INFINITY && x0 >= -kSureRange));
                        if (good && (!any || in_range)) {
                            bx = any ? m : bx;
                            idx = any ? aw0 + js : idx;
                        } else {
                            m = m0;
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                uint32_t v;
                                asm volatile("mov.b32 %0, %1;" : "=r"(v) : "r"(cur[j]));
                                limb_column(__fadd_rn(__uint_as_float(v), bcur[j]), aw0 + j);
                            }
                        }
                        return;
                    }
                    const float m0 = m, bx0 = bx;
                    const int idx0 = idx;
                    bool bad = false;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        // columns outside [j_lo, j_hi) are masked by their (uniform) predicate, not branched around: the
                        // eight columns stay one basic block
                        const bool act = kFull || (j >= j_lo && j < j_hi);
                        const float x = __fadd_rn(__uint_as_float(cur[j]), bcur[j]);
                        const float d = __fsub_rn(x, m);
                        const bool fast = act && d > kSureStep && fabsf(x) <= kSureRange;
                        bad |= act && !(d <= 0.0f || fast);                 // NaN differences land here too
                        idx = fast ? aw0 + j : idx;
                        bx = fast ? x : bx;
                        m = fmaxf(m, act ? x : -INFINITY);
                    }
                    if (bad) {
                        // (the values pass through an opaque move: otherwise the compiler computes this block's NaN tests
                        // and selects for all eight columns ABOVE the branch, 32 instructions per group)
                        m = m0; bx = bx0; idx = idx0;
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (kFull || (j >= j_lo && j < j_hi)) {
                                uint32_t v;
                                asm volatile("mov.b32 %0, %1;" : "=r"(v) : "r"(cur[j]));
                                limb_column(__fadd_rn(__uint_as_float(v), bcur[j]), aw0 + j);
                            }
                    }
                };
                begin(r_lo);
                int c0 = r_lo;
#pragma unroll 1
                while (c0 < r_hi) {
                    if (limb && !emit && c0 + 8 <= seg_end) {
                        // whole groups inside the current piece: the hot loop
                        // (tried: two register sets, ping-pong, the next group's accumulator columns and bias loaded while this
                        //  group is scanned — 56 bytes of spills at the 96 registers ptxas settles on, cfg2 f16 185 -> 190 us,
                        //  native 346 -> 356 us; the other warps of the scheduler cover the TMEM latency)
#pragma unroll 1
                        do {
                            load_group(c0, cur, bcur);
                            tmem_ld8_wait(cur);
                            spec_scan(std::true_type{}, cur, bcur, 0, 8, c0 - wbase);
                            c0 += 8;
                        } while (c0 + 8 <= seg_end);
                        if (c0 == seg_end) {
                            publish_piece(key0 + (size_t)ei * a.HW, bx, idx, valid);
                            if (seg_end < r_hi) begin(seg_end);
                        }
                        continue;
                    }
                    // a group that holds a piece boundary, decode channels, the ragged end of the run, or any group of a call
                    // that also emits the logits / the head tensor: piece by piece, columns [j_lo, j_hi) at a time
                    load_group(c0, cur, bcur);
                    tmem_ld8_wait(cur);
                    int j_lo = 0;
#pragma unroll 1
                    do {
                        const int j_hi = min(8, seg_end - c0);              // seg_end <= r_hi
                        const int aw0 = c0 - wbase;
                        if (limb && !emit) {
                            spec_scan(std::false_type{}, cur, bcur, j_lo, j_hi, aw0);
                        } else {
                            if (!limb)                                      // decode channels: the logit now, its sigmoid in the finalize pass
                                decode_group(a.dec, b, c0, cell, a.HW, a.n_dec, cur[0], cur[1], cur[2], cur[3], cur[4], cur[5], cur[6], cur[7],
                                             bcur[0], bcur[1], bcur[2], bcur[3], bcur[4], bcur[5], bcur[6], bcur[7], j_lo, j_hi, valid);
                            if (emit) {
#pragma unroll
                                for (int j = 0; j < 8; ++j)
                                    if (j >= j_lo && j < j_hi) {
                                        const float x = __fadd_rn(__uint_as_float(cur[j]), bcur[j]);
                                        emit_column(a.emit_logits, a.emit_head, b, c0 + j, cell, a.C, a.HW, x, valid);
                                        if (limb) limb_column(x, aw0 + j);
                                    }
                            }
                        }
                        j_lo = j_hi;
                        if (c0 + j_hi == seg_end) {
                            if (limb) publish_piece(key0 + (size_t)ei * a.HW, bx, idx, valid);
                            if (seg_end < r_hi) begin(seg_end);
                        }
                    } while (j_lo < 8 && c0 + j_lo < r_hi);
                    c0 += 8;
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
            if (++acc == a.acc_stages) { acc = 0; acc_phase ^= 1u; }
        }
    }
}

// keys -> the uint16 arg-max map (low half of a key = ~position); decode logits -> their sigmoid, in place
__global__ void __launch_bounds__(256)
head_finalize_kernel(const unsigned long long* __restrict__ keys, uint16_t* __restrict__ amax, size_t n_keys, float* __restrict__ dec, size_t n_dec) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_keys) amax[i] = (uint16_t)(0xFFFFFFFFu - (uint32_t)keys[i]);
    if (i < n_dec) dec[i] = sigmoid_f32(dec[i]);
}

// instruction descriptor: D fp32; formats 0 = f16, 1 = bf16, 2 = tf32; bit 15 / 16: A / B MN-major; N >> 3; M >> 4
__device__ __forceinline__ uint32_t mma_idesc(uint32_t fmt, uint32_t a_mn_major, int n) {
    return (1u << 4) | (fmt << 7) | (fmt << 10) | (a_mn_major << 15) | (0u << 16) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(kBlockM >> 4) << 24);
}

// ------------------------------ TF32 path: fp32 NCHW activations read in place ------------------------------
template <int kSubs>
__global__ void __launch_bounds__(64 + 128 * kSubs, 1)
head_gemm_argmax_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w,
                        const __grid_constant__ CUtensorMap tm_wt, HeadArgs a, int pdl) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)kStages * kStageBytes);
    uint64_t* empty = full + kStages;
    uint64_t* tfull = empty + kStages;       // [2] accumulator ready for the epilogue
    uint64_t* tempty = tfull + 2;            // [2] accumulator drained
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&tm_x);
        prefetch_tensormap(&tm_w);
        prefetch_tensormap(&tm_wt);
        for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int q = 0; q < 2; ++q) { mbar_init(&tfull[q], 1); mbar_init(&tempty[q], 4 * kSubs); }
        fence_mbar_init();
    }
    if (warp == 1) {                         // the allocating warp also frees
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (pdl & PDL_WAIT_START) pdl_wait();            // the activations may come from the kernel before us
    if (pdl & PDL_TRIGGER) pdl_launch_dependents();  // the parse kernel may become resident (it waits for us at its top)

    if (warp == 0) {
        // ------------------------------ TMA producer ------------------------------
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
                int tile, nt0, nt1;
                head_item(a, item, tile, nt0, nt1);
                int gb[4], gc[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int g = tile * 4 + q;
                    const int b = g / a.groups_per_img;
                    gb[q] = g < a.n_groups ? b : a.B;                   // past the end: an all-zero box
                    gc[q] = g < a.n_groups ? (g - b * a.groups_per_img) * 32 : 0;
                }
                for (int nt = nt0; nt < nt1; ++nt) {
                    const bool last = nt == a.n_ntiles - 1;             // the last channel tile is only n_last channels wide
                    const uint32_t bytes = kABytes + (uint32_t)(last ? a.n_last : kBlockN) * 128u;
                    for (int kb = 0; kb < a.n_kblocks; ++kb) {
                        mbar_wait_sleep(&empty[stage], phase ^ 1u, 100);
                        unsigned char* sa = smem + (size_t)stage * kStageBytes;
                        mbar_arrive_expect_tx(&full[stage], bytes);
#pragma unroll
                        for (int q = 0; q < 4; ++q) tma_load_3d(sa + q * kGroupBytes, &tm_x, gc[q], kb * kBlockK, gb[q], &full[stage]);
                        tma_load_2d(sa + kABytes, last ? &tm_wt : &tm_w, kb * kBlockK, nt * kBlockN, &full[stage]);
                        if (++stage == kStages) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------ MMA issuer ------------------------------
        if (lane == 0) {
            // A/B tf32, A MN-major (cells contiguous), B K-major, M = 128, N = 256 (n_last for the last channel tile)
            const uint32_t idesc_full = mma_idesc(2u, 1u, kBlockN), idesc_last = mma_idesc(2u, 1u, a.n_last);
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
                int tile, nt0, nt1;
                head_item(a, item, tile, nt0, nt1);
                for (int nt = nt0; nt < nt1; ++nt) {
                    const uint32_t idesc = nt == a.n_ntiles - 1 ? idesc_last : idesc_full;
                    mbar_wait_sleep(&tempty[acc], acc_phase ^ 1u, 40);   // the epilogue has drained this accumulator
                    tc_fence_after();
                    const uint32_t d = tmem_base + (uint32_t)acc * kBlockN;
                    for (int kb = 0; kb < a.n_kblocks; ++kb) {
                        mbar_wait_sleep(&full[stage], phase, 20);
                        tc_fence_after();
                        const uint32_t sa = smem_u32(smem + (size_t)stage * kStageBytes), sb = sa + kABytes;
#pragma unroll
                        for (int kk = 0; kk < kBlockK / kUmmaK; ++kk) {
                            // A (MN-major): k-rows of 128 B (32 cells), swizzle atoms of 4 rows (512 B), 8 rows per
                            //    instruction, cell groups 4096 B apart;
                            // B (K-major): 8 channel rows of 128 B per atom (1024 B), K advanced by 32 B inside the row
                            const uint64_t da = smem_desc(sa + kk * 1024, kGroupBytes, 512, 1);
                            const uint64_t db = smem_desc(sb + kk * kUmmaK * 4, 16, 1024, 2);
                            tc_mma<0>(d, da, db, idesc, (kb | kk) != 0 ? 1u : 0u);
                        }
                        tc_commit(&empty[stage]);                        // the stage is free once these MMAs have read it
                        if (++stage == kStages) { stage = 0; phase ^= 1u; }
                    }
                    tc_commit(&tfull[acc]);
                    if (++acc == a.acc_stages) { acc = 0; acc_phase ^= 1u; }
                }
            }
        }
    } else {
        head_epilogue<kSubs, false>(a, tmem_base, tfull, tempty);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// ------------------------------ 16-bit path: packed K-major operands ------------------------------
// Activations [B * HW][Cin] and weights [C][Cin] in fp16 or bf16, both K-major (input channels contiguous: what
// head_pack_kernel writes, or a channels_last 16-bit tensor of the network itself), kind::f16 MMAs at twice the TF32
// rate on half the operand bytes.  A tile is 128 consecutive rows of the flattened (image, cell) list — no padding
// of H*W to a multiple of 32 — and its activations (Cin <= 512: at most 128 KB) are loaded ONCE and stay in shared
// memory for all channel tiles; only the weights stream through a ring.  Each k-block slot of the resident A tile has
// its own full/empty barrier pair, so the next tile's activations stream in right behind the last channel tile's
// sweep over the slots instead of after it.
constexpr int kBlockK16 = 64;                // 16-bit elements per 128-byte swizzle row
constexpr int kUmmaK16 = 16;
constexpr int kMaxKBlocks16 = 8;             // Cin <= 512
constexpr int kA16Bytes = kBlockM * 128;     // one k-block of the A tile: 16 KB
constexpr int kMaxBStages = 12;              // stages of the weight ring: acc_n rows of 128 bytes each (16 KB at 128 channels)
constexpr int kMaxAcc16 = 4;                 // accumulators: 4 x 128 columns (or 2 x 256)
constexpr int kBar16Bytes = 512;

template <int kSubs>
__global__ void __launch_bounds__(64 + 128 * kSubs, 1)
head_gemm16_argmax_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w,
                          const __grid_constant__ CUtensorMap tm_wt, HeadArgs a, int pdl) {
    extern __shared__ __align__(1024) unsigned char smem16[];
    unsigned char* sA = smem16;                                               // [n_kblocks][16 KB]
    unsigned char* sB = smem16 + (size_t)a.n_kblocks * kA16Bytes;             // [n_bstages][32 KB]
    const uint32_t b_stage_bytes = (uint32_t)a.acc_n * 128u;                   // one stage of the weight ring: acc_n rows of one k-block
    uint64_t* afull = reinterpret_cast<uint64_t*>(sB + (size_t)a.n_bstages * b_stage_bytes);
    uint64_t* aempty = afull + kMaxKBlocks16;
    uint64_t* bfull = aempty + kMaxKBlocks16;
    uint64_t* bempty = bfull + kMaxBStages;
    uint64_t* tfull = bempty + kMaxBStages;
    uint64_t* tempty = tfull + kMaxAcc16;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + kMaxAcc16);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (warp == 0 && lane == 0) {
        if (smem_u32(smem16) & 1023u) __trap();      // the 128-byte swizzle atoms need the 1024-byte alignment asked for
        prefetch_tensormap(&tm_x);
        prefetch_tensormap(&tm_w);
        prefetch_tensormap(&tm_wt);
        for (int s = 0; s < kMaxKBlocks16; ++s) { mbar_init(&afull[s], 1); mbar_init(&aempty[s], 1); }
        for (int s = 0; s < kMaxBStages; ++s) { mbar_init(&bfull[s], 1); mbar_init(&bempty[s], 1); }
        for (int q = 0; q < kMaxAcc16; ++q) { mbar_init(&tfull[q], 1); mbar_init(&tempty[q], 4 * kSubs); }
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (pdl & PDL_WAIT_START) pdl_wait();            // the packed operands come from the kernel before us
    if (pdl & PDL_TRIGGER) pdl_launch_dependents();

    if (warp == 0) {
        // ------------------------------ TMA producer ------------------------------
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, a_phase = 0;
            for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
                int tile, nt0, nt1;
                head_item(a, item, tile, nt0, nt1);
                for (int nt = nt0; nt < nt1; ++nt) {
                    const bool last = nt == a.n_ntiles - 1;
                    const uint32_t b_bytes = (uint32_t)(last ? a.n_last : a.acc_n) * 128u;
                    for (int kb = 0; kb < a.n_kblocks; ++kb) {
                        if (nt == nt0) {                                 // this item's activations, k-block by k-block
                            mbar_wait_sleep(&aempty[kb], a_phase ^ 1u, 100);
                            mbar_arrive_expect_tx(&afull[kb], kA16Bytes);
                            tma_load_2d(sA + (size_t)kb * kA16Bytes, &tm_x, kb * kBlockK16, tile * kBlockM, &afull[kb]);
                        }
                        mbar_wait_sleep(&bempty[stage], phase ^ 1u, 100);
                        mbar_arrive_expect_tx(&bfull[stage], b_bytes);
                        tma_load_2d(sB + (size_t)stage * b_stage_bytes, last ? &tm_wt : &tm_w, kb * kBlockK16, nt * a.acc_n, &bfull[stage]);
                        if (++stage == a.n_bstages) { stage = 0; phase ^= 1u; }
                    }
                }
                a_phase ^= 1u;
            }
        }
    } else if (warp == 1) {
        // ------------------------------ MMA issuer ------------------------------
        if (lane == 0) {
            const uint32_t fmt = a.bf16 ? 1u : 0u;
            const uint32_t idesc_full = mma_idesc(fmt, 0u, a.acc_n), idesc_last = mma_idesc(fmt, 0u, a.n_last);
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0, a_phase = 0;
            for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
                int tile, nt0, nt1;
                head_item(a, item, tile, nt0, nt1);
                for (int nt = nt0; nt < nt1; ++nt) {
                    const bool last = nt == a.n_ntiles - 1, last_of_item = nt == nt1 - 1;
                    const uint32_t idesc = last ? idesc_last : idesc_full;
                    mbar_wait_sleep(&tempty[acc], acc_phase ^ 1u, 40);
                    tc_fence_after();
                    const uint32_t d = tmem_base + (uint32_t)(acc * a.acc_n);
                    for (int kb = 0; kb < a.n_kblocks; ++kb) {
                        if (nt == nt0) mbar_wait_sleep(&afull[kb], a_phase, 20);
                        mbar_wait_sleep(&bfull[stage], phase, 20);
                        tc_fence_after();
                        const uint32_t sa = smem_u32(sA + (size_t)kb * kA16Bytes), sb = smem_u32(sB + (size_t)stage * b_stage_bytes);
#pragma unroll
                        for (int kk = 0; kk < kBlockK16 / kUmmaK16; ++kk) {
                            // both K-major: 8 rows of 128 B per swizzle atom (1024 B), K advanced by 32 B inside the row
                            const uint64_t da = smem_desc(sa + kk * kUmmaK16 * 2, 16, 1024, 2);
                            const uint64_t db = smem_desc(sb + kk * kUmmaK16 * 2, 16, 1024, 2);
                            if (!(a.dry & 2) || kb == 0) tc_mma<1>(d, da, db, idesc, (kb | kk) != 0 ? 1u : 0u);
                        }
                        tc_commit(&bempty[stage]);
                        if (last_of_item) tc_commit(&aempty[kb]);        // the next item's k-block may land here
                        if (++stage == a.n_bstages) { stage = 0; phase ^= 1u; }
                    }
                    tc_commit(&tfull[acc]);
                    if (++acc == a.acc_stages) { acc = 0; acc_phase ^= 1u; }
                }
                a_phase ^= 1u;
            }
        }
    } else {
        head_epilogue<kSubs, true>(a, tmem_base, tfull, tempty);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// ------------------------------ operand packing for the 16-bit path ------------------------------
// feat [B][Cin][HW] fp32 (NCHW) -> xt [B * HW][Cin] T (round to nearest even), weight [C][Cin] fp32 -> wt [C][Cin] T.
// Blocks [0, n_feat_blocks): one 64-channel x 32-cell tile each, transposed through shared memory (128-byte reads along
// the cells, 128-byte writes along the channels); the blocks after them convert the weights.  (narrow / bits16:
// ppn_device.cuh)
template <typename T>
__global__ void __launch_bounds__(256)
head_pack_kernel(const float* __restrict__ feat, const float* __restrict__ weight, T* __restrict__ xt, T* __restrict__ wt,
                 int Cin, int HW, int chunks_per_img, int kchunks, int n_feat_blocks, size_t n_weight) {
    __shared__ float tile[64][33];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if ((int)blockIdx.x < n_feat_blocks) {
        const int kc = blockIdx.x % kchunks;
        const int t = blockIdx.x / kchunks;
        const int b = t / chunks_per_img, cc = t - b * chunks_per_img;
        const int cell = cc * 32 + lane;
        const float* src = feat + ((size_t)b * Cin + (size_t)kc * 64) * HW;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = cell < HW ? __ldg(src + (size_t)(warp * 8 + i) * HW + cell) : 0.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) tile[warp * 8 + i][lane] = v[i];
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int cl = warp * 4 + i, c = cc * 32 + cl;
            if (c < HW) {
                const uint32_t pair = bits16(narrow<T>(tile[2 * lane][cl])) | (bits16(narrow<T>(tile[2 * lane + 1][cl])) << 16);
                *reinterpret_cast<uint32_t*>(xt + ((size_t)b * HW + c) * Cin + (size_t)kc * 64 + 2 * lane) = pair;
            }
        }
    } else {
        const size_t n4 = n_weight / 4;
        const size_t stride = (size_t)(gridDim.x - n_feat_blocks) * blockDim.x;
        for (size_t i = (size_t)(blockIdx.x - n_feat_blocks) * blockDim.x + threadIdx.x; i < n4; i += stride) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(weight) + i);
            *reinterpret_cast<uint2*>(wt + 4 * i) = make_uint2(bits16(narrow<T>(w.x)) | (bits16(narrow<T>(w.y)) << 16),
                                                                bits16(narrow<T>(w.z)) | (bits16(narrow<T>(w.w)) << 16));
        }
    }
}

// ---- host side ----------------------------------------------------------------------------------------
namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
std::mutex g_enc_mu;
EncodeTiledFn g_encode = nullptr;
bool g_attr_done[64] = {};

cudaError_t encoder(EncodeTiledFn* out) {
    std::lock_guard<std::mutex> lock(g_enc_mu);
    if (!g_encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
        if (e != cudaSuccess) return e;
        if (q != cudaDriverEntryPointSuccess || !fn) return cudaErrorNotSupported;
        g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    *out = g_encode;
    return cudaSuccess;
}

// 2-D row-major matrix [rows][cols] of `elem_bytes`-wide elements, box = box_cols x box_rows, 128-byte swizzle
bool map_2d(EncodeTiledFn enc, CUtensorMap* m, CUtensorMapDataType dt, int elem_bytes, const void* base, uint64_t cols, uint64_t rows,
            uint32_t box_cols, uint32_t box_rows) {
    const cuuint64_t dim[2] = {cols, rows};
    const cuuint64_t stride[1] = {cols * (uint64_t)elem_bytes};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t es[2] = {1, 1};
    return enc(m, dt, 2, const_cast<void*>(base), dim, stride, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

size_t head16_smem_bytes(int n_kblocks, int n_bstages, int acc_n) {
    return (size_t)n_kblocks * kA16Bytes + (size_t)n_bstages * acc_n * 128 + kBar16Bytes;
}

void fill_common(HeadArgs& a, const Geom& g, int Cin, const float* bias, float* dec, unsigned long long* keys, float* emit_logits, float* emit_head,
                 int acc_n = kBlockN) {
    a.B = g.B; a.HW = g.HW; a.Cin = Cin; a.C = g.C; a.n_dec = 6 * g.K; a.S = g.S; a.E = g.E;
    a.acc_n = acc_n; a.acc_stages = kTmemCols / acc_n;
    a.n_ntiles = (g.C + acc_n - 1) / acc_n;
    a.n_last = ((g.C - (a.n_ntiles - 1) * acc_n) + 15) & ~15;              // 16 .. acc_n
    a.magic_S = g.S <= 1 ? 0u : (uint32_t)(((1ull << 32) + g.S - 1) / g.S);
    a.bias = bias; a.dec = dec; a.keys = keys; a.emit_logits = emit_logits; a.emit_head = emit_head;
    a.n_rows = g.B * g.HW; a.n_bstages = 0; a.bf16 = 0; a.dry = 0;
    a.groups_per_img = (g.HW + 31) / 32;
    a.n_groups = g.B * a.groups_per_img;
}
template <bool k16, int kSubs>
cudaError_t launch_gemm_n(int grid, size_t smem, cudaStream_t st, bool pdl_attr, const CUtensorMap& tm_x, const CUtensorMap& tm_w,
                          const CUtensorMap& tm_wt, const HeadArgs& a, int pdl_bits) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(64 + 128 * kSubs);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_attr ? 1 : 0;
    if constexpr (k16) return cudaLaunchKernelEx(&cfg, head_gemm16_argmax_kernel<kSubs>, tm_x, tm_w, tm_wt, a, pdl_bits);
    else return cudaLaunchKernelEx(&cfg, head_gemm_argmax_kernel<kSubs>, tm_x, tm_w, tm_wt, a, pdl_bits);
}
// epilogue warps per TMEM lane quadrant: instantiated for 1, 2, 4 and 6 (3 runs as 4, 5 and 7 as 6)
template <bool k16>
cudaError_t launch_gemm(int subs, int grid, size_t smem, cudaStream_t st, bool pdl_attr, const CUtensorMap& tm_x, const CUtensorMap& tm_w,
                        const CUtensorMap& tm_wt, const HeadArgs& a, int pdl_bits) {
    if (subs <= 1) return launch_gemm_n<k16, 1>(grid, smem, st, pdl_attr, tm_x, tm_w, tm_wt, a, pdl_bits);
    if (subs == 2) return launch_gemm_n<k16, 2>(grid, smem, st, pdl_attr, tm_x, tm_w, tm_wt, a, pdl_bits);
    if (subs <= 4) return launch_gemm_n<k16, 4>(grid, smem, st, pdl_attr, tm_x, tm_w, tm_wt, a, pdl_bits);
    return launch_gemm_n<k16, 6>(grid, smem, st, pdl_attr, tm_x, tm_w, tm_wt, a, pdl_bits);
}
template <bool k16, int kSubs>
cudaError_t set_smem_attr_n(int bytes) {
    if constexpr (k16) return cudaFuncSetAttribute(head_gemm16_argmax_kernel<kSubs>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    else return cudaFuncSetAttribute(head_gemm_argmax_kernel<kSubs>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
template <bool k16>
cudaError_t set_smem_attr(int bytes) {
    cudaError_t e;
    if ((e = set_smem_attr_n<k16, 1>(bytes)) != cudaSuccess) return e;
    if ((e = set_smem_attr_n<k16, 2>(bytes)) != cudaSuccess) return e;
    if ((e = set_smem_attr_n<k16, 4>(bytes)) != cudaSuccess) return e;
    return set_smem_attr_n<k16, 6>(bytes);
}
cudaError_t finalize_amax(const unsigned long long* keys, uint16_t* amax, float* dec, const Geom& g, cudaStream_t st) {
    const size_t n_keys = (size_t)g.B * g.E * g.HW, n_dec = (size_t)g.B * 6 * g.K * g.HW, n = std::max(n_keys, n_dec);
    if (n == 0) return cudaSuccess;
    head_finalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(keys, amax, n_keys, dec, n_dec);
    return cudaGetLastError();
}
// Fewer cell tiles than SMs (small batches — one image of the reference's shape is 5 tiles): cut every cell tile's channel
// tiles into chunks, one work item each, so that about one item lands on every SM.  The pieces of a limb window meet in
// the key maxima wherever they were scanned, so nothing else changes; a CTA re-loads its activations per item.
void plan_items(HeadArgs& a, int sms) {
    int chunks = 1;
    if (a.n_tiles < sms) chunks = std::min(a.n_ntiles, std::max(1, sms / a.n_tiles));
    a.chunk_tiles = (a.n_ntiles + chunks - 1) / chunks;
    a.n_chunks = (a.n_ntiles + a.chunk_tiles - 1) / a.chunk_tiles;
    a.n_items = a.n_tiles * a.n_chunks;
}
}  // namespace

size_t head_keys_bytes(const Geom& g) { return (size_t)g.B * g.E * g.HW * sizeof(unsigned long long); }

size_t head_smem_bytes() { return (size_t)kStages * kStageBytes + 1024 /* alignment slack */ + 256 /* barriers, TMEM slot */; }

cudaError_t launch_head_gemm_argmax(const float* feat, const float* weight, const float* bias, int Cin, const Geom& g,
                                    float* dec, uint16_t* amax, unsigned long long* keys, float* emit_logits, float* emit_head,
                                    cudaStream_t st, bool pdl_attr, int pdl_bits, int subs) {
    if (g.B == 0) return cudaSuccess;
    if (Cin % kBlockK != 0 || g.HW % 4 != 0) return cudaErrorInvalidValue;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    EncodeTiledFn enc = nullptr;
    if ((e = encoder(&enc)) != cudaSuccess) return e;

    HeadArgs a;
    fill_common(a, g, Cin, bias, dec, keys, emit_logits, emit_head);
    a.dry = (subs >> 8) & 3;
    subs &= 255;
    if (subs == 0) subs = 4;
    a.n_tiles = (a.n_groups + 3) / 4;
    a.n_kblocks = Cin / kBlockK;
    plan_items(a, sms);

    CUtensorMap tm_x, tm_w, tm_wt;
    {   // activations [B][Cin][HW] fp32: box = 32 cells x 32 input channels of one image
        const cuuint64_t dim[3] = {(cuuint64_t)g.HW, (cuuint64_t)Cin, (cuuint64_t)g.B};
        const cuuint64_t stride[2] = {(cuuint64_t)g.HW * 4, (cuuint64_t)Cin * g.HW * 4};
        const cuuint32_t box[3] = {32, (cuuint32_t)kBlockK, 1};
        const cuuint32_t es[3] = {1, 1, 1};
        if (enc(&tm_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(feat), dim, stride, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    // weights [C][Cin] fp32: box = 32 input channels x 256 output channels (x n_last for the last channel tile)
    if (!map_2d(enc, &tm_w, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, weight, Cin, g.C, kBlockK, kBlockN) ||
        !map_2d(enc, &tm_wt, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, weight, Cin, g.C, kBlockK, a.n_last))
        return cudaErrorInvalidValue;

    const size_t smem = head_smem_bytes();
    {
        std::lock_guard<std::mutex> lock(g_enc_mu);
        if (dev >= 0 && dev < 64 && !g_attr_done[dev]) {
            if ((e = set_smem_attr<false>((int)smem)) != cudaSuccess) return e;
            g_attr_done[dev] = true;
        }
    }
    if ((e = cudaMemsetAsync(keys, 0, head_keys_bytes(g), st)) != cudaSuccess) return e;
    if ((e = launch_gemm<false>(subs, std::min(sms, a.n_items), smem, st, pdl_attr, tm_x, tm_w, tm_wt, a, pdl_bits)) != cudaSuccess) return e;
    return finalize_amax(keys, amax, dec, g, st);
}

bool head16_supported(int Cin, const Geom& g) {
    return Cin >= kBlockK16 && Cin % kBlockK16 == 0 && Cin <= kMaxKBlocks16 * kBlockK16 && (long long)g.B * g.HW < (1ll << 31) - kBlockM;
}

size_t head16_packed_feat_bytes(int Cin, const Geom& g) { return (size_t)g.B * g.HW * Cin * 2; }
size_t head16_packed_weight_bytes(int Cin, const Geom& g) { return (size_t)g.C * Cin * 2; }

// feat: fp32 NCHW when `feat_nchw_f32` (packed into `xt` first), else 16-bit [B * HW][Cin] in the operand type, used in place
cudaError_t launch_head_gemm16_argmax(const void* feat, bool feat_nchw_f32, const float* weight, const float* bias, int Cin, bool bf16,
                                      const Geom& g, void* xt, void* wt, float* dec, uint16_t* amax, unsigned long long* keys,
                                      float* emit_logits, float* emit_head, cudaStream_t st, int pdl_bits, int subs) {
    if (g.B == 0) return cudaSuccess;
    if (!head16_supported(Cin, g)) return cudaErrorInvalidValue;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    EncodeTiledFn enc = nullptr;
    if ((e = encoder(&enc)) != cudaSuccess) return e;

    HeadArgs a;
    // accumulators: two of 256 channels.  (tune key head.acc = 128: four of 128 channels, the weight ring in 16 KB stages —
    // meant to give the MMA side and the epilogue more slack around each other; measured, it halves the work per barrier
    // round trip of the one MMA-issuing thread instead: operand stream + MMAs alone 212 -> 375 us at the native shape, the
    // whole kernel 299 -> 438 us.  Parity-green, kept as a knob.)
    const int acc_n = ((subs >> 12) & 1) ? 128 : 256;
    fill_common(a, g, Cin, bias, dec, keys, emit_logits, emit_head, acc_n);
    a.dry = (subs >> 8) & 3;
    subs &= 255;
    if (subs == 0) subs = 6;                  // measured, whole call f16: cfg2 185 -> 181 us, cfg3 672 -> 647, native 355 -> 351 (TF32: 4 stays better)
    a.n_tiles = (a.n_rows + kBlockM - 1) / kBlockM;
    a.n_kblocks = Cin / kBlockK16;
    plan_items(a, sms);
    a.bf16 = bf16 ? 1 : 0;
    int max_smem = 0;
    if ((e = cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
    a.n_bstages = kMaxBStages;
    while (a.n_bstages > 2 && head16_smem_bytes(a.n_kblocks, a.n_bstages, acc_n) > (size_t)max_smem) --a.n_bstages;
    const size_t smem = head16_smem_bytes(a.n_kblocks, a.n_bstages, acc_n);
    if (smem > (size_t)max_smem) return cudaErrorInvalidValue;

    if ((e = cudaMemsetAsync(keys, 0, head_keys_bytes(g), st)) != cudaSuccess) return e;
    // 1. pack: activations (unless they already are K-major 16-bit) and weights
    {
        const int chunks = (g.HW + 31) / 32, kchunks = Cin / 64;
        const int n_feat_blocks = feat_nchw_f32 ? g.B * chunks * kchunks : 0;
        const size_t n_weight = (size_t)g.C * Cin;
        const int n_w_blocks = (int)std::min<size_t>((n_weight / 4 + 255) / 256, 4 * (size_t)sms);
        const float* f32 = feat_nchw_f32 ? static_cast<const float*>(feat) : nullptr;
        if (bf16)
            head_pack_kernel<__nv_bfloat16><<<n_feat_blocks + n_w_blocks, 256, 0, st>>>(f32, weight, static_cast<__nv_bfloat16*>(xt), static_cast<__nv_bfloat16*>(wt),
                                                                                        Cin, g.HW, chunks, kchunks, n_feat_blocks, n_weight);
        else
            head_pack_kernel<__half><<<n_feat_blocks + n_w_blocks, 256, 0, st>>>(f32, weight, static_cast<__half*>(xt), static_cast<__half*>(wt),
                                                                                 Cin, g.HW, chunks, kchunks, n_feat_blocks, n_weight);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    // 2. GEMM + epilogue
    const void* x16 = feat_nchw_f32 ? xt : feat;
    const CUtensorMapDataType dt = bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    CUtensorMap tm_x, tm_w, tm_wt;
    if (!map_2d(enc, &tm_x, dt, 2, x16, Cin, (uint64_t)a.n_rows, kBlockK16, kBlockM) ||
        !map_2d(enc, &tm_w, dt, 2, wt, Cin, g.C, kBlockK16, acc_n) ||
        !map_2d(enc, &tm_wt, dt, 2, wt, Cin, g.C, kBlockK16, a.n_last))
        return cudaErrorInvalidValue;
    {
        std::lock_guard<std::mutex> lock(g_enc_mu);
        static bool done16[64] = {};
        if (dev >= 0 && dev < 64 && !done16[dev]) {
            if ((e = set_smem_attr<true>(max_smem)) != cudaSuccess) return e;
            done16[dev] = true;
        }
    }
    // its prologue (barriers, TMEM, tensor maps) runs under the pack kernel's tail
    if ((e = launch_gemm<true>(subs, std::min(sms, a.n_items), smem, st, true, tm_x, tm_w, tm_wt, a, pdl_bits | PDL_WAIT_START)) != cudaSuccess) return e;
    return finalize_amax(keys, amax, dec, g, st);
}

}  // namespace ppn
