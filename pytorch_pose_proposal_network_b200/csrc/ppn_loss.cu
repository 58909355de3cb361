// PPNLoss (the reference's criterion, main.py:125-216) as two fused kernels over the head tensor and the
// encoded targets, hand-written for sm_100a.
//
// The loss of one image, for head channels resp, conf, x, y, w, h (K each) and the limb block e [E, sH, sW, H, W]
// (specification: the float64 restatement of the test infrastructure, ppn_loss.py; DESIGN.md §11 says which points of it are
// reconstructed rather than pinned to the reference):
//   L_resp = sum (resp - delta)^2                 L_iou  = sum delta (conf - iou)^2
//   L_coor = sum weight ((x - tx_half)^2 + (y - ty_half)^2)
//   L_size = sum weight ((sqrt(w + eps) - sqrt(tw + eps))^2 + (sqrt(h + eps) - sqrt(th + eps))^2)
//   L_limb = sum weight_ij (e - te)^2
// each averaged over the batch (sum / B); eps = 1e-6 (config.EPSILON).
//
// Work is split into ITEMS, handed out statically (CTA c takes items c, c + grid, ...):
//   small items   1024 cells of the [B, K, H, W] planes: a thread takes whole cells, because the IoU needs all four
//                 box planes of a cell (6 head values and 8 targets in, 4 loss terms or 6 gradients out);
//   limb items    8192 consecutive elements of one image's limb block, streamed with 128-bit loads (and, backward,
//                 128-bit streaming stores) from the first element at which the head, te, weight_ij (and grad) of
//                 that image all sit on a 16-byte boundary, element by element where no such element exists (only
//                 grids with an odd H*W or odd K produce such images, or tensors whose storage starts mid-vector).
// The limb block is 98.6 % of the bytes at the native shape: the kernels are HBM streams with a little arithmetic.
//
// Element types (the AMP setup of the reference, main.py:282-289): the head, and with it the gradient, may be fp16 or
// bf16; te and weight_ij then may be fp32 or the head's type; the eight small targets are always fp32.  A 16-bit
// element is widened to fp32 exactly when it is loaded, everything below is the fp32 arithmetic as written, and a
// gradient element is rounded once, to nearest even, to the head's type when it is stored (overflow gives +-inf, as
// torch's .to() does; a GradScaler looks for it).  So a 16-bit run equals the fp32 run on the widened inputs followed
// by .to(head.dtype).  With a 16-bit stream a vector step covers 8 elements: one 16-byte access per 16-bit stream,
// two per fp32 stream.
//
// Forward: every thread accumulates its terms in fp64 (each fp32 term converted exactly); a CTA reduces its threads
// in a fixed butterfly order and stores 5 doubles into the caller's workspace; a one-CTA kernel sums the CTA
// partials in a fixed order and writes loss[t] = (float)(sum_t / B).  No float atomics: the same inputs on the same
// device give the same bits.
//
// Backward: recomputes everything from the inputs (nothing is saved by the forward) and writes every element of
// grad_head once.  fp32, one rounding per operation (__f*_rn, no FMA contraction; the build also has -fmad=false),
// in exactly this order (grad_model_f32 of the test infrastructure is the same sequence in numpy float32):
//   with g = grad_loss[5] (device) and Bf = (float)B:
//     cr = (2 * g0) / Bf   ci = (2 * g1) / Bf   cc = (2 * g2) / Bf   cs = g3 / Bf   cl = (2 * g4) / Bf
//   limb     grad = cl * (weight_ij * (e - te))
//   resp     grad = cr * (resp - delta)
//   IoU of the cell (column X, row Y as floats):
//     px = (x + X) * gW   py = (y + Y) * gH   pw = inW * w   ph = inH * h      (q.. likewise from tx, ty, tw, th)
//     px1 = px - pw * 0.5   px2 = px + pw * 0.5   (qx1, qx2, py1, ... likewise)
//     iwr = min(px2, qx2) - max(px1, qx1)   iw = iwr > 0 ? iwr : 0          (ihr, ih likewise in y)
//     I = iw * ih   U = ((pw * ph + qw * qh) - I) + eps   iou = I / U
//   conf     a = ci * (delta * (conf - iou));  grad = a
//   IoU chain, from diou = -a:
//     r = diou / U   ri = r * iou   dI = r + ri                                 (d iou/dI = 1/U + I/U^2)
//     giw = iwr > 0 ? dI * ih : 0   gih = ihr > 0 ? dI * iw : 0                 (relu'(0) = 0)
//     s2 = px2 < qx2 ? 1 : px2 == qx2 ? 0.5 : 0   s1 = px1 > qx1 ? 1 : px1 == qx1 ? 0.5 : 0   (ties split evenly)
//     dpx2 = giw * s2   dpx1 = -(giw * s1)   dpx = dpx2 + dpx1   dpw = (dpx2 - dpx1) * 0.5 - ri * ph
//     (y: the same with gih, py*, qy*; dph = (dpy2 - dpy1) * 0.5 - ri * pw)
//   x        grad = cc * (weight * (x - tx_half)) + dpx * gW                    (y likewise with ty_half, dpy, gH)
//   w        sw = sqrt(w + eps)   st = sqrt(tw + eps);  grad = cs * (weight * ((sw - st) / sw)) + dpw * inW
//                                                                               (h likewise with th, dph, inH)
// min / max are fminf / fmaxf: the inputs are taken to be finite (a NaN head is not a training state).
//
// From logits (kLogits, the *_logits exports): the head holds the conv output x before the network's sigmoid
// (model.py:133-136), for every channel.  Each head element is widened as above and replaced at once by
// s = sigmoid_f32(x) (ppn_device.cuh: libdevice expf, one add, one IEEE division; +-inf gives 0 or 1); everything
// above runs on s, operation for operation, and s is never narrowed.  A gradient element g_s (fp32, before any
// narrowing) becomes
//   grad_x = (g_s * (1 - s)) * s                                                 (torch's sigmoid_backward)
// and only then is stored, rounded once to the head's type.  The sigmoid-input instantiations (kLogits = false)
// compile to what they were before this path existed.
#include <algorithm>
#include <atomic>

#include "ppn_kernels.h"

namespace ppn {

namespace {

constexpr int kLossThreads = 256;
constexpr int kSmallCells = 1024;      // cells of the [B, K, H, W] planes per small item
constexpr int kLimbChunk = 8192;       // limb elements per limb item: 32 KB of each fp32 stream
constexpr int kLimbUnroll = 4;         // vector steps whose loads a thread issues before it computes
constexpr int kLogitsUnroll = 1;       // the same on logits: the sigmoid makes them issue-bound, and 1 (48-62 registers,
                                       // 4+ CTAs per SM) measured 7-19 % faster per kernel than 4 (DESIGN.md §11)
constexpr float kEps = 1e-6f;          // config.EPSILON

// ---- streaming element access (no L1 allocation), widened to / narrowed from fp32 ------------------------------
__device__ __forceinline__ float lds(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ unsigned short lds16(const void* p) {
    unsigned short v;
    asm volatile("ld.global.nc.L1::no_allocate.b16 %0, [%1];" : "=h"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ldw(const float* p) { return lds(p); }
__device__ __forceinline__ float ldw(const __half* p) { return widen(__ushort_as_half(lds16(p))); }
__device__ __forceinline__ float ldw(const __nv_bfloat16* p) { return widen(__ushort_as_bfloat16(lds16(p))); }

__device__ __forceinline__ void st16(void* p, unsigned short v) { asm volatile("st.global.cs.b16 [%0], %1;" ::"l"(p), "h"(v) : "memory"); }
__device__ __forceinline__ void stw(float* p, float v) { __stcs(p, v); }
__device__ __forceinline__ void stw(__half* p, float v) { st16(p, __half_as_ushort(narrow<__half>(v))); }
__device__ __forceinline__ void stw(__nv_bfloat16* p, float v) { st16(p, __bfloat16_as_ushort(narrow<__nv_bfloat16>(v))); }

// ---- 16-byte vectors: VE consecutive elements of one stream kept as raw words, widened when used -----------------
__device__ __forceinline__ uint4 ldg_stream_u4(const void* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t word(const uint4& q, int k) { return k == 0 ? q.x : k == 1 ? q.y : k == 2 ? q.z : q.w; }
__device__ __forceinline__ unsigned short half_word(const uint4* q, int i) {
    const uint32_t w = word(q[i >> 3], (i >> 1) & 3);
    return (unsigned short)((i & 1) ? (w >> 16) : (w & 0xffffu));
}

template <typename T, int VE> struct Vec {
    uint4 q[VE * (int)sizeof(T) / 16];
    __device__ __forceinline__ void load(const T* p) {                // p: 16-byte aligned
#pragma unroll
        for (int i = 0; i < VE * (int)sizeof(T) / 16; ++i) q[i] = ldg_stream_u4(reinterpret_cast<const uint4*>(p) + i);
    }
};
template <int VE> __device__ __forceinline__ float at(const Vec<float, VE>& v, int i) { return __uint_as_float(word(v.q[i >> 2], i & 3)); }
template <int VE> __device__ __forceinline__ float at(const Vec<__half, VE>& v, int i) { return widen(__ushort_as_half(half_word(v.q, i))); }
template <int VE> __device__ __forceinline__ float at(const Vec<__nv_bfloat16, VE>& v, int i) {
    return widen(__ushort_as_bfloat16(half_word(v.q, i)));
}

// VE gradients (p: 16-byte aligned) with 128-bit streaming stores
template <int VE> __device__ __forceinline__ void st_vec(float* p, const float (&g)[VE]) {
#pragma unroll
    for (int j = 0; j < VE / 4; ++j) __stcs(reinterpret_cast<float4*>(p) + j, make_float4(g[4 * j], g[4 * j + 1], g[4 * j + 2], g[4 * j + 3]));
}
template <typename T, int VE> __device__ __forceinline__ void st_vec(T* p, const float (&g)[VE]) {    // 16-bit types
#pragma unroll
    for (int j = 0; j < VE / 8; ++j)
        __stcs(reinterpret_cast<uint4*>(p) + j, make_uint4(pack2<T>(g[8 * j], g[8 * j + 1]), pack2<T>(g[8 * j + 2], g[8 * j + 3]),
                                                           pack2<T>(g[8 * j + 4], g[8 * j + 5]), pack2<T>(g[8 * j + 6], g[8 * j + 7])));
}

// elements of a vector step: 4 when every stream is fp32, else 8
template <typename TH, typename TL> __host__ __device__ constexpr int vec_elems() { return sizeof(TH) == 4 && sizeof(TL) == 4 ? 4 : 8; }

struct Cell {
    float resp, conf, x, y, w, h;                           // head
    float delta, weight, txh, tyh, tx, ty, tw, th;          // targets
};

// a head element as the loss uses it: the widened value, or its sigmoid when the head holds logits
template <bool kLogits> __device__ __forceinline__ float act(float v) {
    if constexpr (kLogits) return sigmoid_f32(v); else return v;
}
// the gradient of the stored head element from g, the gradient of the value act() gave (s)
template <bool kLogits> __device__ __forceinline__ float chain(float g, float s) {
    if constexpr (kLogits) return __fmul_rn(__fmul_rn(g, __fsub_rn(1.0f, s)), s); else return g;
}

template <typename TH, bool kLogits>
__device__ __forceinline__ Cell load_cell(const LossArgs& a, long long i) {
    const long long KHW = (long long)a.K * a.HW;
    const long long b = i / KHW, r = i - b * KHW;
    const TH* img = static_cast<const TH*>(a.head) + (size_t)b * a.img_stride + (size_t)r;
    const size_t KH = (size_t)KHW;
    Cell c;
    c.resp = act<kLogits>(ldw(img));          c.conf = act<kLogits>(ldw(img + KH));     c.x = act<kLogits>(ldw(img + 2 * KH));
    c.y = act<kLogits>(ldw(img + 3 * KH));    c.w = act<kLogits>(ldw(img + 4 * KH));    c.h = act<kLogits>(ldw(img + 5 * KH));
    c.delta = lds(a.delta + i); c.weight = lds(a.weight + i);
    c.txh = lds(a.tx_half + i); c.tyh = lds(a.ty_half + i);
    c.tx = lds(a.tx + i);       c.ty = lds(a.ty + i);       c.tw = lds(a.tw + i);       c.th = lds(a.th + i);
    return c;
}

struct Box {
    float p1, p2, q1, q2;       // predicted / target interval along one axis
    float size, qsize, r, i;    // predicted / target extent (pw, qw or ph, qh), raw and relu'd intersection
};

__device__ __forceinline__ Box axis(float v, float t, float sz, float tsz, float pos, float grid, float in) {
    Box o;
    const float p = __fmul_rn(__fadd_rn(v, pos), grid), q = __fmul_rn(__fadd_rn(t, pos), grid);
    o.size = __fmul_rn(in, sz);
    o.qsize = __fmul_rn(in, tsz);
    const float hp = __fmul_rn(o.size, 0.5f), hq = __fmul_rn(o.qsize, 0.5f);
    o.p1 = __fsub_rn(p, hp); o.p2 = __fadd_rn(p, hp);
    o.q1 = __fsub_rn(q, hq); o.q2 = __fadd_rn(q, hq);
    o.r = __fsub_rn(fminf(o.p2, o.q2), fmaxf(o.p1, o.q1));
    o.i = o.r > 0.0f ? o.r : 0.0f;
    return o;
}

struct Iou { Box x, y; float I, U, iou; };

__device__ __forceinline__ Iou iou_of(const LossArgs& a, const Cell& c, long long i) {
    const int cell = (int)(i % a.HW);
    const int row = cell / a.W, col = cell - row * a.W;
    Iou o;
    o.x = axis(c.x, c.tx, c.w, c.tw, (float)col, a.gW, a.inW);
    o.y = axis(c.y, c.ty, c.h, c.th, (float)row, a.gH, a.inH);
    o.I = __fmul_rn(o.x.i, o.y.i);
    o.U = __fadd_rn(__fsub_rn(__fadd_rn(__fmul_rn(o.x.size, o.y.size), __fmul_rn(o.x.qsize, o.y.qsize)), o.I), kEps);
    o.iou = __fdiv_rn(o.I, o.U);
    return o;
}

// d(loss)/d(p1), d(loss)/d(p2) of one axis and the resulting gradient of its position and extent (before the
// area term), from the gradient `gi` of the relu'd intersection
__device__ __forceinline__ void axis_grad(const Box& b, float gi, float* d_pos, float* d_size_half) {
    const float s2 = b.p2 < b.q2 ? 1.0f : (b.p2 == b.q2 ? 0.5f : 0.0f);
    const float s1 = b.p1 > b.q1 ? 1.0f : (b.p1 == b.q1 ? 0.5f : 0.0f);
    const float d2 = __fmul_rn(gi, s2);
    const float d1 = -__fmul_rn(gi, s1);
    *d_pos = __fadd_rn(d2, d1);
    *d_size_half = __fmul_rn(__fsub_rn(d2, d1), 0.5f);
}

__device__ __forceinline__ float sq(float v) { return __fmul_rn(v, v); }

// ---- the limb block of one item ---------------------------------------------------------------------------------
template <typename TH, typename TL> struct LimbItem { const TH* hp; const TL *tp, *wp; TH* gp; int start, end, pro; bool vec; };

__device__ __forceinline__ bool on_16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <typename TH, typename TL>
__device__ __forceinline__ LimbItem<TH, TL> limb_item(const LossArgs& a, long long j, bool backward) {
    const long long b = j / a.limb_chunks;
    const int q = (int)(j - b * a.limb_chunks);
    LimbItem<TH, TL> it;
    it.hp = static_cast<const TH*>(a.head) + (size_t)b * a.img_stride + a.limb_off;
    it.tp = static_cast<const TL*>(a.te) + (size_t)b * a.L;
    it.wp = static_cast<const TL*>(a.weight_ij) + (size_t)b * a.L;
    it.gp = backward ? static_cast<TH*>(a.grad) + (size_t)b * a.img_stride + a.limb_off : nullptr;
    // The head has the most elements per 16 bytes of any stream (8 if 16-bit, else 4 like all the others), so the
    // first element at which every stream is 16-byte aligned, if there is one, is the head's first aligned element.
    const int h0 = (int)(((16u - (reinterpret_cast<uintptr_t>(it.hp) & 15u)) & 15u) / sizeof(TH));
    it.vec = on_16(it.tp + h0) && on_16(it.wp + h0) && (!backward || on_16(it.gp + h0));
    const int a0 = it.vec ? min(a.L, h0) : 0;                           // elements before the first aligned vector
    it.pro = q == 0 ? a0 : 0;                                            // chunk 0 also takes those
    it.start = min(a.L, a0 + q * kLimbChunk);
    it.end = min(a.L, it.start + kLimbChunk);
    return it;
}

__device__ __forceinline__ float limb_term(float e, float t, float w) { return __fmul_rn(w, sq(__fsub_rn(e, t))); }
__device__ __forceinline__ float limb_grad(float cl, float e, float t, float w) {
    return __fmul_rn(cl, __fmul_rn(w, __fsub_rn(e, t)));
}
// the same from the stored head element h
template <bool kLogits> __device__ __forceinline__ float limb_term_at(float h, float t, float w) {
    return limb_term(act<kLogits>(h), t, w);
}
template <bool kLogits> __device__ __forceinline__ float limb_grad_at(float cl, float h, float t, float w) {
    const float e = act<kLogits>(h);
    return chain<kLogits>(limb_grad(cl, e, t, w), e);
}

// deterministic CTA sum of 5 doubles; thread 0..4 store the CTA's partials
__device__ __forceinline__ void cta_store(double acc[5], double* out) {
    __shared__ double s[kLossThreads / 32][5];
#pragma unroll
    for (int t = 0; t < 5; ++t)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[t] += __shfl_xor_sync(0xffffffffu, acc[t], o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0)
#pragma unroll
        for (int t = 0; t < 5; ++t) s[warp][t] = acc[t];
    __syncthreads();
    if (threadIdx.x < 5) {
        double v = 0.0;
        for (int w = 0; w < kLossThreads / 32; ++w) v += s[w][threadIdx.x];
        out[(size_t)blockIdx.x * 5 + threadIdx.x] = v;
    }
}

template <typename TH, typename TL, bool kLogits>
__global__ void __launch_bounds__(kLossThreads)
loss_forward_kernel(LossArgs a) {
    constexpr int VE = vec_elems<TH, TL>();
    constexpr int UN = kLogits ? kLogitsUnroll : kLimbUnroll;
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    const int tid = threadIdx.x;
    const long long n_cells = (long long)a.B * a.K * a.HW;
    for (long long j = blockIdx.x; j < a.n_items; j += gridDim.x) {
        if (j < a.small_items) {
            const long long c1 = min(n_cells, (j + 1) * kSmallCells);
            for (long long i = j * kSmallCells + tid; i < c1; i += kLossThreads) {
                const Cell c = load_cell<TH, kLogits>(a, i);
                const Iou u = iou_of(a, c, i);
                acc[0] += (double)sq(__fsub_rn(c.resp, c.delta));
                acc[1] += (double)__fmul_rn(c.delta, sq(__fsub_rn(c.conf, u.iou)));
                acc[2] += (double)__fmul_rn(c.weight, __fadd_rn(sq(__fsub_rn(c.x, c.txh)), sq(__fsub_rn(c.y, c.tyh))));
                const float dw = __fsub_rn(__fsqrt_rn(__fadd_rn(c.w, kEps)), __fsqrt_rn(__fadd_rn(c.tw, kEps)));
                const float dh = __fsub_rn(__fsqrt_rn(__fadd_rn(c.h, kEps)), __fsqrt_rn(__fadd_rn(c.th, kEps)));
                acc[3] += (double)__fmul_rn(c.weight, __fadd_rn(sq(dw), sq(dh)));
            }
            continue;
        }
        const LimbItem<TH, TL> it = limb_item<TH, TL>(a, j - a.small_items, false);
        if (tid < it.pro) acc[4] += (double)limb_term_at<kLogits>(ldw(it.hp + tid), ldw(it.tp + tid), ldw(it.wp + tid));
        int s0 = it.start;
        if (it.vec) {
            const int nv = (it.end - it.start) / VE;
            for (int v0 = tid; v0 < nv; v0 += UN * kLossThreads) {
                Vec<TH, VE> hv[UN];
                Vec<TL, VE> tv[UN], wv[UN];
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    const size_t e = (size_t)it.start + (size_t)(v0 + u * kLossThreads) * VE;
                    if (v0 + u * kLossThreads < nv) { hv[u].load(it.hp + e); tv[u].load(it.tp + e); wv[u].load(it.wp + e); }
                }
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    if (v0 + u * kLossThreads < nv) {
#pragma unroll
                        for (int k = 0; k < VE; ++k) acc[4] += (double)limb_term_at<kLogits>(at(hv[u], k), at(tv[u], k), at(wv[u], k));
                    }
                }
            }
            s0 = it.start + VE * nv;
        }
        for (int e = s0 + tid; e < it.end; e += kLossThreads)             // vector tail, or the whole unaligned item
            acc[4] += (double)limb_term_at<kLogits>(ldw(it.hp + e), ldw(it.tp + e), ldw(it.wp + e));
    }
    cta_store(acc, a.partial);
}

// loss[t] = (float)(sum over CTAs of partial[cta][t] / B): warp t sums term t, lanes in a fixed stride, then a
// fixed butterfly
__global__ void __launch_bounds__(160)
loss_finalize_kernel(const double* __restrict__ partial, int n, int B, float* __restrict__ loss) {
    const int t = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double v = 0.0;
    for (int i = lane; i < n; i += 32) v += partial[(size_t)i * 5 + t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) loss[t] = (float)(v / (double)B);
}

template <typename TH, typename TL, bool kLogits>
__global__ void __launch_bounds__(kLossThreads)
loss_backward_kernel(LossArgs a) {
    constexpr int VE = vec_elems<TH, TL>();
    constexpr int UN = kLogits ? kLogitsUnroll : kLimbUnroll;
    const float Bf = (float)a.B;
    const float cr = __fdiv_rn(__fmul_rn(2.0f, a.grad_loss[0]), Bf);
    const float ci = __fdiv_rn(__fmul_rn(2.0f, a.grad_loss[1]), Bf);
    const float cc = __fdiv_rn(__fmul_rn(2.0f, a.grad_loss[2]), Bf);
    const float cs = __fdiv_rn(a.grad_loss[3], Bf);
    const float cl = __fdiv_rn(__fmul_rn(2.0f, a.grad_loss[4]), Bf);
    const int tid = threadIdx.x;
    const long long n_cells = (long long)a.B * a.K * a.HW;
    const long long KHW = (long long)a.K * a.HW;
    for (long long j = blockIdx.x; j < a.n_items; j += gridDim.x) {
        if (j < a.small_items) {
            const long long c1 = min(n_cells, (j + 1) * kSmallCells);
            for (long long i = j * kSmallCells + tid; i < c1; i += kLossThreads) {
                const Cell c = load_cell<TH, kLogits>(a, i);
                const Iou u = iou_of(a, c, i);
                const float g_resp = __fmul_rn(cr, __fsub_rn(c.resp, c.delta));
                const float g_conf = __fmul_rn(ci, __fmul_rn(c.delta, __fsub_rn(c.conf, u.iou)));
                const float diou = -g_conf;
                const float r = __fdiv_rn(diou, u.U);
                const float ri = __fmul_rn(r, u.iou);
                const float dI = __fadd_rn(r, ri);
                const float giw = u.x.r > 0.0f ? __fmul_rn(dI, u.y.i) : 0.0f;
                const float gih = u.y.r > 0.0f ? __fmul_rn(dI, u.x.i) : 0.0f;
                float dpx, dpw, dpy, dph;
                axis_grad(u.x, giw, &dpx, &dpw);
                axis_grad(u.y, gih, &dpy, &dph);
                dpw = __fsub_rn(dpw, __fmul_rn(ri, u.y.size));
                dph = __fsub_rn(dph, __fmul_rn(ri, u.x.size));
                const float g_x = __fadd_rn(__fmul_rn(cc, __fmul_rn(c.weight, __fsub_rn(c.x, c.txh))), __fmul_rn(dpx, a.gW));
                const float g_y = __fadd_rn(__fmul_rn(cc, __fmul_rn(c.weight, __fsub_rn(c.y, c.tyh))), __fmul_rn(dpy, a.gH));
                const float sw = __fsqrt_rn(__fadd_rn(c.w, kEps)), st = __fsqrt_rn(__fadd_rn(c.tw, kEps));
                const float sh = __fsqrt_rn(__fadd_rn(c.h, kEps)), sth = __fsqrt_rn(__fadd_rn(c.th, kEps));
                const float g_w = __fadd_rn(__fmul_rn(cs, __fmul_rn(c.weight, __fdiv_rn(__fsub_rn(sw, st), sw))), __fmul_rn(dpw, a.inW));
                const float g_h = __fadd_rn(__fmul_rn(cs, __fmul_rn(c.weight, __fdiv_rn(__fsub_rn(sh, sth), sh))), __fmul_rn(dph, a.inH));
                const long long b = i / KHW, rr = i - b * KHW;
                TH* gimg = static_cast<TH*>(a.grad) + (size_t)b * a.img_stride + (size_t)rr;
                const size_t KH = (size_t)KHW;
                stw(gimg, chain<kLogits>(g_resp, c.resp));       stw(gimg + KH, chain<kLogits>(g_conf, c.conf));
                stw(gimg + 2 * KH, chain<kLogits>(g_x, c.x));    stw(gimg + 3 * KH, chain<kLogits>(g_y, c.y));
                stw(gimg + 4 * KH, chain<kLogits>(g_w, c.w));    stw(gimg + 5 * KH, chain<kLogits>(g_h, c.h));
            }
            continue;
        }
        const LimbItem<TH, TL> it = limb_item<TH, TL>(a, j - a.small_items, true);
        if (tid < it.pro) stw(it.gp + tid, limb_grad_at<kLogits>(cl, ldw(it.hp + tid), ldw(it.tp + tid), ldw(it.wp + tid)));
        int s0 = it.start;
        if (it.vec) {
            const int nv = (it.end - it.start) / VE;
            for (int v0 = tid; v0 < nv; v0 += UN * kLossThreads) {
                Vec<TH, VE> hv[UN];
                Vec<TL, VE> tv[UN], wv[UN];
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    const size_t e = (size_t)it.start + (size_t)(v0 + u * kLossThreads) * VE;
                    if (v0 + u * kLossThreads < nv) { hv[u].load(it.hp + e); tv[u].load(it.tp + e); wv[u].load(it.wp + e); }
                }
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    if (v0 + u * kLossThreads < nv) {
                        float g[VE];
#pragma unroll
                        for (int k = 0; k < VE; ++k) g[k] = limb_grad_at<kLogits>(cl, at(hv[u], k), at(tv[u], k), at(wv[u], k));
                        st_vec(it.gp + (size_t)it.start + (size_t)(v0 + u * kLossThreads) * VE, g);
                    }
                }
            }
            s0 = it.start + VE * nv;
        }
        for (int e = s0 + tid; e < it.end; e += kLossThreads)
            stw(it.gp + e, limb_grad_at<kLogits>(cl, ldw(it.hp + e), ldw(it.tp + e), ldw(it.wp + e)));
    }
}

// resident CTAs per SM of each kernel: a property of the compiled kernel, asked once per process
int grid_for(const void* kernel, std::atomic<int>* per_sm_cache, long long n_items, int sms) {
    int per_sm = per_sm_cache->load(std::memory_order_relaxed);
    if (per_sm < 1) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kLossThreads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
        per_sm_cache->store(per_sm, std::memory_order_relaxed);
    }
    return (int)std::min<long long>(n_items, std::min<long long>((long long)sms * per_sm, kLossMaxCtas));
}

template <typename TH, typename TL, bool kLogits>
cudaError_t forward_as(const LossArgs& a, float* loss, int sms, cudaStream_t st) {
    static std::atomic<int> per_sm{0};
    const int grid = grid_for((const void*)loss_forward_kernel<TH, TL, kLogits>, &per_sm, a.n_items, sms);
    loss_forward_kernel<TH, TL, kLogits><<<grid, kLossThreads, 0, st>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    loss_finalize_kernel<<<1, 160, 0, st>>>(a.partial, grid, a.B, loss);
    return cudaGetLastError();
}

template <typename TH, typename TL, bool kLogits>
cudaError_t backward_as(const LossArgs& a, int sms, cudaStream_t st) {
    static std::atomic<int> per_sm{0};
    const int grid = grid_for((const void*)loss_backward_kernel<TH, TL, kLogits>, &per_sm, a.n_items, sms);
    loss_backward_kernel<TH, TL, kLogits><<<grid, kLossThreads, 0, st>>>(a);
    return cudaGetLastError();
}

// the five (head, limb target) type pairs of LossArgs; the C ABI rejects every other pair before launching
template <bool kLogits>
cudaError_t forward_for(const LossArgs& a, float* loss, int sms, cudaStream_t st) {
    switch (a.head_dtype * 3 + a.limb_dtype) {
        case HEAD_F32 * 3 + HEAD_F32: return forward_as<float, float, kLogits>(a, loss, sms, st);
        case HEAD_F16 * 3 + HEAD_F32: return forward_as<__half, float, kLogits>(a, loss, sms, st);
        case HEAD_F16 * 3 + HEAD_F16: return forward_as<__half, __half, kLogits>(a, loss, sms, st);
        case HEAD_BF16 * 3 + HEAD_F32: return forward_as<__nv_bfloat16, float, kLogits>(a, loss, sms, st);
        case HEAD_BF16 * 3 + HEAD_BF16: return forward_as<__nv_bfloat16, __nv_bfloat16, kLogits>(a, loss, sms, st);
        default: return cudaErrorInvalidValue;
    }
}

template <bool kLogits>
cudaError_t backward_for(const LossArgs& a, int sms, cudaStream_t st) {
    switch (a.head_dtype * 3 + a.limb_dtype) {
        case HEAD_F32 * 3 + HEAD_F32: return backward_as<float, float, kLogits>(a, sms, st);
        case HEAD_F16 * 3 + HEAD_F32: return backward_as<__half, float, kLogits>(a, sms, st);
        case HEAD_F16 * 3 + HEAD_F16: return backward_as<__half, __half, kLogits>(a, sms, st);
        case HEAD_BF16 * 3 + HEAD_F32: return backward_as<__nv_bfloat16, float, kLogits>(a, sms, st);
        case HEAD_BF16 * 3 + HEAD_BF16: return backward_as<__nv_bfloat16, __nv_bfloat16, kLogits>(a, sms, st);
        default: return cudaErrorInvalidValue;
    }
}

// ppn_sigmoid: the sigmoid the loss applies, elementwise into fp32 (grid-stride; not a hot path)
template <typename T>
__global__ void __launch_bounds__(256) sigmoid_kernel(const T* __restrict__ x, float* __restrict__ y, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        y[i] = sigmoid_f32(widen(x[i]));
}

}  // namespace

void loss_plan(LossArgs* a) {
    const long long n_cells = (long long)a->B * a->K * a->HW;
    a->small_items = (n_cells + kSmallCells - 1) / kSmallCells;
    a->limb_chunks = a->L > 0 ? (a->L + kLimbChunk - 1) / kLimbChunk : 0;
    a->n_items = a->small_items + (long long)a->B * a->limb_chunks;
}

size_t loss_workspace_bytes(const LossArgs& a) {
    const long long ctas = std::min<long long>(std::max<long long>(a.n_items, 1), kLossMaxCtas);
    return (size_t)ctas * 5 * sizeof(double);
}

cudaError_t launch_loss_forward(LossArgs a, float* loss, int sms, cudaStream_t st, bool from_logits) {
    return from_logits ? forward_for<true>(a, loss, sms, st) : forward_for<false>(a, loss, sms, st);
}

cudaError_t launch_loss_backward(LossArgs a, int sms, cudaStream_t st, bool from_logits) {
    return from_logits ? backward_for<true>(a, sms, st) : backward_for<false>(a, sms, st);
}

cudaError_t launch_sigmoid(const void* x, int dtype, float* y, size_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const int grid = (int)std::min<size_t>((n + 255) / 256, 8192);
    switch (dtype) {
        case HEAD_F32: sigmoid_kernel<<<grid, 256, 0, st>>>(static_cast<const float*>(x), y, n); break;
        case HEAD_F16: sigmoid_kernel<<<grid, 256, 0, st>>>(static_cast<const __half*>(x), y, n); break;
        case HEAD_BF16: sigmoid_kernel<<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), y, n); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

}  // namespace ppn
