// Proposal-pair parse (ppn_parse_proposals), stage 2: limb scores of candidate pairs and the greedy tree parse in
// which humans compete for parts.  Stage 1 is decode_nms_kernel with n_parts = K (ppn_kernels.cu): it leaves the
// NMS survivors of every (image, part) in the workspace.  The rule is specified in DESIGN.md §13.
//
// One CTA per image.  Shared memory holds the humans' part cells and, for the limb being matched, the cell -> state
// maps of its source and target part; nothing is stored per pair.  The greedy matching (pairs by score descending,
// then human, then cell; accept when both ends are free) equals the matching built by rounds of "mutually best"
// pairs: a pair that is the best available pair of its human AND of its target cell under that strict total order
// is accepted by the sequential rule, whatever else is accepted in the same round.  So each round
//   A  recomputes the best available target of every human whose previous best was taken,
//   B  recomputes the best available human of every target cell whose previous best was matched,
//   C  accepts every pair that is the best of both of its ends,
//   D  marks the bests that C made stale,
// and the limb is done when a round accepts nothing (then no available pair is left: the best of all would be
// mutual).  A best is a 64-bit key: the score's bits (sc > 0, so they order like the floats) above the complement of
// the other end's index (the smaller index wins a tie).  A and B evaluate a pair's score with the same fp32
// operations, so the two ends agree on its key bit for bit.
#include <algorithm>

#include "ppn_kernels.h"

namespace ppn {

namespace {

constexpr int kPairThreads = 256;
constexpr unsigned long long kStale = ~0ull;     // best must be recomputed (a score key never has all bits set)

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w > v ? w : v;
    }
    return v;
}

// (delta_s * lv) * delta_t, left to right, one rounding each; 0 unless sc > 0 (NaN, 0 and negatives never connect)
__device__ __forceinline__ unsigned long long pair_key(float ds, float lv, float dt, unsigned other) {
    const float sc = __fmul_rn(__fmul_rn(ds, lv), dt);
    return sc > 0.0f ? ((unsigned long long)__float_as_uint(sc) << 32) | (0xFFFFFFFFu - other) : 0ull;
}

struct PairSmem {
    unsigned long long* best_h;   // [HW] per human: key of its best available target (0: none, kStale: recompute)
    unsigned long long* best_t;   // [HW] per target cell: key of its best available human
    float* t_delta;               // [HW] delta of the target part at each of its proposals
    float* s_delta;               // [HW] per human: delta of its source-part cell
    int16_t* cell;                // [HW][K] part cells of every human (-1 = absent); human i = i-th root proposal
    int16_t* owner;               // [HW] cell -> human holding the source part there (-1); reused as slot -> human
    uint8_t* t_free;              // [HW] 1: a proposal of the target part that no human holds yet
};

// carve the dynamic shared memory of one CTA (16-byte aligned blocks); s == nullptr: only the size
__host__ __device__ inline size_t pair_smem_layout(int HW, int K, PairSmem* s, unsigned char* base) {
    const size_t hw = (size_t)HW;
    auto up = [](size_t v) { return (v + 15) & ~(size_t)15; };
    const size_t o_best_t = up(hw * 8), o_t_delta = o_best_t + up(hw * 8), o_s_delta = o_t_delta + up(hw * 4);
    const size_t o_cell = o_s_delta + up(hw * 4), o_owner = o_cell + up(hw * K * 2), o_t_free = o_owner + up(hw * 2);
    if (s) {
        s->best_h = reinterpret_cast<unsigned long long*>(base);
        s->best_t = reinterpret_cast<unsigned long long*>(base + o_best_t);
        s->t_delta = reinterpret_cast<float*>(base + o_t_delta);
        s->s_delta = reinterpret_cast<float*>(base + o_s_delta);
        s->cell = reinterpret_cast<int16_t*>(base + o_cell);
        s->owner = reinterpret_cast<int16_t*>(base + o_owner);
        s->t_free = base + o_t_free;
    }
    return o_t_free + up(hw);
}

template <typename T>
__global__ void __launch_bounds__(kPairThreads, 4)
proposal_pairs_kernel(const T* __restrict__ head, Geom g, LimbTree tree, int min_kp,
                      const int32_t* __restrict__ keep_cell, const int32_t* __restrict__ keep_count,
                      int32_t* __restrict__ h_count, int32_t* __restrict__ h_root, int32_t* __restrict__ h_cell,
                      float* __restrict__ h_score, float4* __restrict__ h_box, int R) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_acc[2];
    __shared__ int warp_tot[kPairThreads / 32];
    __shared__ int base_s;
    PairSmem s;
    pair_smem_layout(g.HW, g.K, &s, smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n_warps = blockDim.x >> 5;
    const int HW = g.HW, K = g.K, W = g.W;
    const int b = blockIdx.x;
    const T* img = head + (size_t)b * g.img_stride;
    const T* lmb = img + g.limb_off;
    // a programmatic dependent of decode + NMS: the proposal lists are complete only past this wait
    pdl_wait();
    const int32_t* kc = keep_count + (size_t)b * K;
    const int32_t* kl = keep_cell + (size_t)b * K * HW;
    const int n0 = kc[0];
    for (int q = tid; q < n0 * K; q += blockDim.x) {
        const int i = q / K, k = q - i * K;
        s.cell[q] = k == 0 ? (int16_t)kl[i] : (int16_t)-1;
    }
    for (int q = 0; q < tree.n; ++q) {
        const int e = tree.limb[q], src = tree.src[q], t = tree.dst[q];
        const int nt = kc[t];
        const int32_t* Pt = kl + (size_t)t * HW;
        const T* lmb_e = lmb + (size_t)e * g.S * HW;
        __syncthreads();                                             // previous limb (or the root fill) complete
        for (int c = tid; c < HW; c += blockDim.x) { s.t_free[c] = 0; s.owner[c] = -1; s.best_t[c] = 0; }
        if (tid == 0) s_acc[0] = s_acc[1] = 0;
        __syncthreads();
        for (int j = tid; j < nt; j += blockDim.x) {
            const int c = Pt[j];
            s.t_free[c] = 1;
            s.t_delta[c] = delta_at(img, g, t, c);
            s.best_t[c] = kStale;
        }
        for (int i = tid; i < n0; i += blockDim.x) {
            const int a = s.cell[i * K + src];
            if (a >= 0) { s.owner[a] = (int16_t)i; s.s_delta[i] = delta_at(img, g, src, a); s.best_h[i] = kStale; }
            else s.best_h[i] = 0;
        }
        __syncthreads();
        for (int round = 0;; ++round) {
            // A: a warp per stale human, its lanes over the window positions; only available targets are gathered
            for (int i = warp; i < n0; i += n_warps) {
                if (s.best_h[i] != kStale) continue;                 // warp-uniform
                const int a = s.cell[i * K + src];
                const int ih = a / W, iw = a - ih * W;
                const float ds = s.s_delta[i];
                unsigned long long best = 0;
                for (int p = lane; p < g.S; p += 32) {
                    const int dy = p / g.sW, dx = p - dy * g.sW;
                    const int jh = ih + dy - g.off_h, jw = iw + dx - g.off_w;
                    if (jh < 0 || jh >= g.H || jw < 0 || jw >= W) continue;
                    const int c = jh * W + jw;
                    if (!s.t_free[c]) continue;
                    const unsigned long long k = pair_key(ds, ldf(lmb_e + (size_t)p * HW + a), s.t_delta[c], (unsigned)c);
                    best = k > best ? k : best;
                }
                best = warp_max_u64(best);
                if (lane == 0) s.best_h[i] = best;
            }
            // B: a warp per stale target, its lanes over the window positions that can reach it
            for (int j = warp; j < nt; j += n_warps) {
                const int c = Pt[j];
                if (s.best_t[c] != kStale) continue;                 // warp-uniform
                const int jh = c / W, jw = c - jh * W;
                const float dt = s.t_delta[c];
                unsigned long long best = 0;
                for (int p = lane; p < g.S; p += 32) {
                    const int dy = p / g.sW, dx = p - dy * g.sW;
                    const int ih = jh - dy + g.off_h, iw = jw - dx + g.off_w;
                    if (ih < 0 || ih >= g.H || iw < 0 || iw >= W) continue;
                    const int a = ih * W + iw;
                    const int i = s.owner[a];
                    if (i < 0 || s.cell[i * K + t] >= 0) continue;
                    const unsigned long long k = pair_key(s.s_delta[i], ldf(lmb_e + (size_t)p * HW + a), dt, (unsigned)i);
                    best = k > best ? k : best;
                }
                best = warp_max_u64(best);
                if (lane == 0) s.best_t[c] = best;
            }
            __syncthreads();
            // C: accept the mutual bests.  A target names one human, so no two threads accept the same cell.
            for (int i = tid; i < n0; i += blockDim.x) {
                const unsigned long long k = s.best_h[i];
                if (k == 0) continue;
                const int c = (int)(0xFFFFFFFFu - (unsigned)k);
                if (s.best_t[c] == ((k & 0xFFFFFFFF00000000ull) | (0xFFFFFFFFu - (unsigned)i))) {
                    s.cell[i * K + t] = (int16_t)c;
                    s.best_h[i] = 0;
                    s.t_free[c] = 0;
                    s.best_t[c] = 0;
                    s_acc[round & 1] = 1;
                }
            }
            __syncthreads();
            if (!s_acc[round & 1]) break;                            // uniform
            if (tid == 0) s_acc[(round + 1) & 1] = 0;                // last read two barriers ago
            // D: bests whose other end was taken in C are recomputed next round
            for (int i = tid; i < n0; i += blockDim.x) {
                const unsigned long long k = s.best_h[i];
                if (k != 0 && !s.t_free[0xFFFFFFFFu - (unsigned)k]) s.best_h[i] = kStale;
            }
            for (int j = tid; j < nt; j += blockDim.x) {
                const int c = Pt[j];
                const unsigned long long k = s.best_t[c];
                if (s.t_free[c] && k != 0 && s.cell[(int)(0xFFFFFFFFu - (unsigned)k) * K + t] >= 0) s.best_t[c] = kStale;
            }
            __syncthreads();
        }
    }
    __syncthreads();
    // humans with at least min_kp non-root parts, in root NMS order: slot -> human in s.owner
    if (tid == 0) base_s = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n0; i0 += blockDim.x) {
        const int i = i0 + tid;
        bool keep = false;
        if (i < n0) {
            int present = 0;
            for (int k = 1; k < K; ++k) present += s.cell[i * K + k] >= 0;
            keep = present >= min_kp;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) warp_tot[warp] = __popc(bal);
        __syncthreads();
        int off = base_s, total = 0;
        for (int w = 0; w < n_warps; ++w) { if (w < warp) off += warp_tot[w]; total += warp_tot[w]; }
        if (keep) s.owner[off + __popc(bal & ((1u << lane) - 1u))] = (int16_t)i;
        __syncthreads();
        if (tid == 0) base_s += total;
        __syncthreads();
    }
    const int n_out = base_s;
    if (tid == 0) h_count[b] = n_out;
    const int used = min(n_out, R);
    for (int j = warp; j < used; j += n_warps) {
        const int i = s.owner[j];
        const size_t slot = (size_t)b * R + j;
        for (int k = lane; k < K; k += 32) {
            const int c = s.cell[i * K + k];
            const size_t o = slot * K + k;
            h_cell[o] = c;
            h_score[o] = c >= 0 ? delta_at(img, g, k, c) : 0.0f;
            h_box[o] = c >= 0 ? box_at(img, g, k, c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (lane == 0) h_root[slot] = s.cell[i * K];
    }
}

struct PairDevice { int smem_optin = 0; size_t granted[3] = {0, 0, 0}; };
PairDevice g_pair_dev[64];

template <typename T>
cudaError_t launch_pairs_t(const cudaLaunchConfig_t& cfg, const T* head, const Geom& g, const LimbTree& tree, int min_kp,
                           const int32_t* keep_cell, const int32_t* keep_count, int32_t* h_count, int32_t* h_root,
                           int32_t* h_cell, float* h_score, float* h_box, int R, size_t smem, size_t* granted) {
    if (smem > *granted) {
        const cudaError_t e = cudaFuncSetAttribute(proposal_pairs_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        *granted = smem;
    }
    return cudaLaunchKernelEx(&cfg, proposal_pairs_kernel<T>, head, g, tree, min_kp, keep_cell, keep_count, h_count, h_root,
                              h_cell, h_score, reinterpret_cast<float4*>(h_box), R);
}

}  // namespace

size_t proposal_pairs_smem_bytes(const Geom& g) { return pair_smem_layout(g.HW, g.K, nullptr, nullptr); }

cudaError_t launch_proposal_pairs(const void* head, const Geom& g, const LimbTree& tree, int min_kp,
                                  const int32_t* keep_cell, const int32_t* keep_count, int32_t* h_count, int32_t* h_root,
                                  int32_t* h_cell, float* h_score, float* h_box, int R, cudaStream_t st) {
    if (g.B == 0) return cudaSuccess;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    PairDevice& d = g_pair_dev[dev];
    if (!d.smem_optin && (e = cudaDeviceGetAttribute(&d.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess)
        return e;
    const size_t smem = proposal_pairs_smem_bytes(g);
    if (smem > (size_t)d.smem_optin) return cudaErrorInvalidConfiguration;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)g.B);
    cfg.blockDim = dim3(kPairThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;    // starts beside decode + NMS, waits inside
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    switch (g.dtype) {
        case HEAD_F32: return launch_pairs_t(cfg, static_cast<const float*>(head), g, tree, min_kp, keep_cell, keep_count, h_count,
                                             h_root, h_cell, h_score, h_box, R, smem, &d.granted[0]);
        case HEAD_F16: return launch_pairs_t(cfg, static_cast<const __half*>(head), g, tree, min_kp, keep_cell, keep_count, h_count,
                                             h_root, h_cell, h_score, h_box, R, smem, &d.granted[1]);
        case HEAD_BF16: return launch_pairs_t(cfg, static_cast<const __nv_bfloat16*>(head), g, tree, min_kp, keep_cell, keep_count,
                                              h_count, h_root, h_cell, h_score, h_box, R, smem, &d.granted[2]);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace ppn
