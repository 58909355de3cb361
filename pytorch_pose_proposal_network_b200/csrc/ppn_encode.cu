// Training-target encoder — the inverse of the parser (dataset.py:98-185), hand-written for sm_100a.
//
// People (box, key points, visibility, part size) -> the grids the loss consumes:
//   delta, tx, ty, tw, th            [B, K, H, W]      a labelled part switches its cell on and stores the
//                                                      offset inside the cell and its box size as fractions
//   te                               [B, E, sH, sW, H, W]  one-hot of the displacement between a limb's two cells
//   weight, tx_half, ty_half         [B, K, H, W]      loss weights / centred offsets derived from delta
//   weight_ij                        [B, E, sH, sW, H, W]  1 where either end of the limb is labelled
//                                                      (max(delta_s at the cell, delta_t at the displaced cell))
// te and weight_ij are the same size as the head's limb block, i.e. > 92 % of all bytes: the kernel is
// WRITE-bound and built around that — every element of the two big tensors is written exactly once with
// 128-bit (64-bit when the two are fp16 / bf16) streaming stores by the CTA that owns its (limb, dy, dx) rows,
// weight_ij computed on the fly from a per-image byte map of delta kept in shared memory; the few one-hots of te
// are set afterwards by the same CTA (ordered by a barrier).  In the reference this is ~70 lines of Python per image inside the DataLoader,
// the O(E*H*W) window loop of dataset.py:155-168 among them.
//
// Exactness (the reference's types: key points fp32 tensors, box float64 tensor, part size a Python float):
//   cell = int(x / gridW)            fp32 division, truncation            dataset.py:125-128
//   tx   = x / gridW - ix            fp32 subtraction                     dataset.py:132
//   tw   = w / inW                   float64 division, rounded to fp32 on the store   dataset.py:134
// People are applied in order, so a later person overwrites an earlier one's cell values (dataset.py:108).
#include <algorithm>

#include "ppn_kernels.h"

namespace ppn {

struct EncPoint { int iy, ix; float fx, fy; bool labeled; };

// part k of person p: is it labelled, which cell does it fall into (dataset.py:112-128)
__device__ __forceinline__ EncPoint enc_point(const EncodeArgs& a, int p, int k) {
    EncPoint r;
    float x, y;
    if (k == 0) {
        const double w = a.bbox[4 * (size_t)p + 2], h = a.bbox[4 * (size_t)p + 3];
        r.labeled = w > 0.0 && h > 0.0;                                  // dataset.py:115
        x = (float)a.bbox[4 * (size_t)p];                                // torch.tensor([cx.item(), cy.item()]) -> fp32
        y = (float)a.bbox[4 * (size_t)p + 1];
    } else {
        r.labeled = a.visible[(size_t)p * (a.K - 1) + (k - 1)] != 0;
        x = a.keypoints[((size_t)p * (a.K - 1) + (k - 1)) * 2];
        y = a.keypoints[((size_t)p * (a.K - 1) + (k - 1)) * 2 + 1];
    }
    r.fx = __fdiv_rn(x, a.gridW);
    r.fy = __fdiv_rn(y, a.gridH);
    r.ix = (int)r.fx;                                                    // int(): towards zero
    r.iy = (int)r.fy;
    return r;
}

// four consecutive limb-tensor elements (p: 16-byte aligned for fp32, 8-byte for 16 bits), one streaming store
__device__ __forceinline__ void st4(float* p, const float (&v)[4]) { __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3])); }
template <typename T> __device__ __forceinline__ void st4(T* p, const float (&v)[4]) {
    __stcs(reinterpret_cast<uint2*>(p), make_uint2(pack2<T>(v[0], v[1]), pack2<T>(v[2], v[3])));
}

// TL: the element type of te and weight_ij (float, __half or __nv_bfloat16); the eight small grids are fp32
template <typename TL>
__global__ void __launch_bounds__(256)
encode_targets_kernel(EncodeArgs a) {
    extern __shared__ __align__(16) unsigned char s_delta[];              // [K * HW] 0 / 1
    const int b = blockIdx.x, z = blockIdx.y;
    const int tid = threadIdx.x, T = blockDim.x;
    const int HW = a.H * a.W, KHW = a.K * HW, S = a.sH * a.sW;
    const int p0 = a.person_off[b], n_p = a.person_off[b + 1] - p0;

    for (int i = tid; i < KHW; i += T) s_delta[i] = 0;
    __syncthreads();
    // ---- delta as a byte map: every labelled part inside the grid (any order) -------------------------
    for (int i = tid; i < n_p * a.K; i += T) {
        const int p = i / a.K, k = i - p * a.K;
        const EncPoint q = enc_point(a, p0 + p, k);
        if (q.labeled && q.iy >= 0 && q.iy < a.H && q.ix >= 0 && q.ix < a.W) s_delta[k * HW + q.iy * a.W + q.ix] = 1;
    }
    __syncthreads();

    // ---- the [K, H, W] grids, by the image's first CTA --------------------------------------------------
    if (z == 0) {
        const size_t base = (size_t)b * KHW;
        for (int i = tid; i < KHW; i += T) {
            a.delta[base + i] = s_delta[i] ? 1.0f : 0.0f;
            a.weight[base + i] = s_delta[i] ? 1.0f : 0.0005f;            // min(delta + 0.0005 [delta < 0.5], 1)  dataset.py:178-180
            if (!s_delta[i]) {
                a.tx[base + i] = 0.0f; a.ty[base + i] = 0.0f; a.tw[base + i] = 0.0f; a.th[base + i] = 0.0f;
                a.tx_half[base + i] = 0.5f; a.ty_half[base + i] = 0.5f;   // 0 + 0.5  dataset.py:182-185
            }
        }
        // values of the switched-on cells: thread k applies the people in order, so the last one wins
        for (int k = tid; k < a.K; k += T) {
            for (int p = 0; p < n_p; ++p) {
                const EncPoint q = enc_point(a, p0 + p, k);
                if (!q.labeled || q.iy < 0 || q.iy >= a.H || q.ix < 0 || q.ix >= a.W) continue;
                const size_t at = base + (size_t)k * HW + q.iy * a.W + q.ix;
                const float ox = __fsub_rn(q.fx, (float)q.ix), oy = __fsub_rn(q.fy, (float)q.iy);
                const double bw = k == 0 ? a.bbox[4 * (size_t)(p0 + p) + 2] : a.size[p0 + p];
                const double bh = k == 0 ? a.bbox[4 * (size_t)(p0 + p) + 3] : a.size[p0 + p];
                a.tx[at] = ox;
                a.ty[at] = oy;
                a.tx_half[at] = ox;                                      // + 0 where delta is set
                a.ty_half[at] = oy;
                a.tw[at] = __double2float_rn(__ddiv_rn(bw, a.inW));
                a.th[at] = __double2float_rn(__ddiv_rn(bh, a.inH));
            }
        }
    }

    if (a.small_only) return;                         // the two limb tensors come from encode_sweep_kernel
    TL* const te = static_cast<TL*>(a.te);
    TL* const weight_ij = static_cast<TL*>(a.weight_ij);
    const float zeros[4] = {0.f, 0.f, 0.f, 0.f};
    // ---- this CTA's rows of te (zeros) and weight_ij, each element written once -------------------------
    const int rows = a.E * S;
    const int r0 = z * a.rows_per_cta, r1 = min(rows, r0 + a.rows_per_cta);
    const size_t big = (size_t)b * rows * HW;
    const int oh = a.sH / 2, ow = a.sW / 2;
    if ((HW & 3) == 0 && (a.W & 3) == 0 && (HW >> 2) <= T) {
        // A thread keeps ONE group of four cells (of one grid row) and walks down the rows of the CTA's
        // range, RL rows apart: its cell coordinates are computed once, the (limb, dy, dx) of a row by an
        // increment and one multiply-high — no integer division in the loop — and both big tensors get one
        // 128-bit streaming store per step.
        const int HW4 = HW >> 2, RL = T / HW4;
        const int lane_r = tid / HW4, c = (tid - lane_r * HW4) << 2;
        if (lane_r < RL) {
            const int h = c / a.W, w = c - h * a.W;
            int r = r0 + lane_r;
            int ei = r / S, wa = r - ei * S;
            for (; r < r1; r += RL) {
                const int dy = a.magic_sW ? (int)__umulhi((unsigned)wa, a.magic_sW) : wa, dx = wa - dy * a.sW;
                const uint32_t ds4 = *reinterpret_cast<const uint32_t*>(s_delta + a.edges.src[ei] * HW + c);   // four source cells
                const unsigned char* dt = s_delta + a.edges.dst[ei] * HW;
                const int hh = h + dy - oh, w0 = w + dx - ow;
                const bool row_in = hh >= 0 && hh < a.H;
                float v[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int ww = w0 + q;
                    const bool on = ((ds4 >> (8 * q)) & 0xffu) || (row_in && ww >= 0 && ww < a.W && dt[hh * a.W + ww]);
                    v[q] = on ? 1.0f : 0.0005f;                          // dataset.py:154-175
                }
                st4(weight_ij + big + (size_t)r * HW + c, v);
                st4(te + big + (size_t)r * HW + c, zeros);
                wa += RL;
                while (wa >= S) { wa -= S; ++ei; }
            }
        }
    } else {
        for (int i = tid; i < (r1 - r0) * HW; i += T) {
            const int r = r0 + i / HW, c = i - (r - r0) * HW;
            const int ei = r / S, w_at = r - ei * S, dy = w_at / a.sW, dx = w_at - dy * a.sW;
            const int h = c / a.W, w = c - h * a.W, hh = h + dy - oh, ww = w + dx - ow;
            const bool on = s_delta[a.edges.src[ei] * HW + c] ||
                            (hh >= 0 && hh < a.H && ww >= 0 && ww < a.W && s_delta[a.edges.dst[ei] * HW + hh * a.W + ww]);
            weight_ij[big + (size_t)r * HW + c] = narrow<TL>(on ? 1.0f : 0.0005f);
            te[big + (size_t)r * HW + c] = narrow<TL>(0.0f);
        }
    }
    __syncthreads();                                  // the zeros of this CTA's rows are ordered before its ones
    // ---- the one-hots of te that fall into this CTA's rows (dataset.py:137-152) --------------------------
    for (int i = tid; i < n_p * a.E; i += T) {
        const int p = i / a.E, ei = i - p * a.E;
        const EncPoint s = enc_point(a, p0 + p, a.edges.src[ei]);
        if (!s.labeled) continue;
        const EncPoint t = enc_point(a, p0 + p, a.edges.dst[ei]);
        if (!t.labeled) continue;
        if (s.iy < 0 || s.ix < 0 || s.iy >= a.H || s.ix >= a.W) continue;
        // (differences of two saturated ints cannot wrap into the window: |int| <= 2^31 - 1, compared in 64 bits)
        const long long jy = (long long)t.iy - s.iy + oh, jx = (long long)t.ix - s.ix + ow;
        if (jy < 0 || jx < 0 || jy >= a.sH || jx >= a.sW) continue;
        const int r = (ei * a.sH + (int)jy) * a.sW + (int)jx;
        if (r >= r0 && r < r1) te[big + (size_t)r * HW + s.iy * a.W + s.ix] = narrow<TL>(1.0f);
    }
}

// The two limb tensors, swept in ADDRESS ORDER by a persistent grid.  A tile is a run of window rows of one
// (image, limb): tiles are numbered in memory order and CTA c takes tiles c, c + grid, ..., so at any moment
// the resident CTAs write one contiguous window of each tensor (a few tens of MB) — the access pattern of a
// plain fill, which is what DRAM write-back wants (with one CTA per (image, half of the rows) there were
// ~1 800 slow write streams spread over the whole tensors: 4.4 TB/s; a fill reaches 6.9).  Per tile the CTA
// rebuilds just the two delta planes it needs (the limb's source and target part) from the image's people.
template <typename TL>
__global__ void __launch_bounds__(256)
encode_sweep_kernel(EncodeArgs a, int B, int chunks, int rows_per_tile) {
    extern __shared__ __align__(16) unsigned char s_planes[];              // [2][HW]: delta of the source / target part
    const int tid = threadIdx.x, T = blockDim.x;
    const int HW = a.H * a.W, S = a.sH * a.sW, HW4 = HW >> 2, RL = T / HW4;
    const int lane_r = tid / HW4, c = (tid - lane_r * HW4) << 2;
    const int h = c / a.W, w = c - h * a.W;
    const int oh = a.sH / 2, ow = a.sW / 2;
    unsigned char* ds = s_planes;
    unsigned char* dt = s_planes + HW;
    TL* const te = static_cast<TL*>(a.te);
    TL* const weight_ij = static_cast<TL*>(a.weight_ij);
    const float zeros[4] = {0.f, 0.f, 0.f, 0.f};
    const long long n_tiles = (long long)B * a.E * chunks;
    for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int ch = (int)(t % chunks);
        const long long be = t / chunks;
        const int ei = (int)(be % a.E), b = (int)(be / a.E);
        const int p0 = a.person_off[b], n_p = a.person_off[b + 1] - p0;
        const int ks = a.edges.src[ei], kt = a.edges.dst[ei];
        __syncthreads();                                                   // the previous tile's planes are dead
        for (int i = tid; i < (2 * HW) >> 2; i += T) reinterpret_cast<uint32_t*>(s_planes)[i] = 0u;
        __syncthreads();
        for (int i = tid; i < 2 * n_p; i += T) {
            const int p = i >> 1, which = i & 1;
            const EncPoint q = enc_point(a, p0 + p, which ? kt : ks);
            if (q.labeled && q.iy >= 0 && q.iy < a.H && q.ix >= 0 && q.ix < a.W) s_planes[which * HW + q.iy * a.W + q.ix] = 1;
        }
        __syncthreads();
        const int wa0 = ch * rows_per_tile, wa1 = min(S, wa0 + rows_per_tile);   // window positions of this tile
        const size_t base = ((size_t)b * a.E + ei) * S * HW;
        if (lane_r < RL) {
            const uint32_t ds4 = *reinterpret_cast<const uint32_t*>(ds + c);       // the four source cells: same for every row
            for (int wa = wa0 + lane_r; wa < wa1; wa += RL) {
                const int dy = a.magic_sW ? (int)__umulhi((unsigned)wa, a.magic_sW) : wa, dx = wa - dy * a.sW;
                const int hh = h + dy - oh, w0 = w + dx - ow;
                const bool row_in = hh >= 0 && hh < a.H;
                float v[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int ww = w0 + q;
                    const bool on = ((ds4 >> (8 * q)) & 0xffu) || (row_in && ww >= 0 && ww < a.W && dt[hh * a.W + ww]);
                    v[q] = on ? 1.0f : 0.0005f;                              // dataset.py:154-175
                }
                st4(weight_ij + base + (size_t)wa * HW + c, v);
                st4(te + base + (size_t)wa * HW + c, zeros);
            }
        }
        __syncthreads();                              // the zeros of this tile are ordered before its ones
        for (int p = tid; p < n_p; p += T) {          // dataset.py:137-152
            const EncPoint s = enc_point(a, p0 + p, ks);
            if (!s.labeled) continue;
            const EncPoint q = enc_point(a, p0 + p, kt);
            if (!q.labeled) continue;
            if (s.iy < 0 || s.ix < 0 || s.iy >= a.H || s.ix >= a.W) continue;
            const long long jy = (long long)q.iy - s.iy + oh, jx = (long long)q.ix - s.ix + ow;
            if (jy < 0 || jx < 0 || jy >= a.sH || jx >= a.sW) continue;
            const int wa = (int)jy * a.sW + (int)jx;
            if (wa >= wa0 && wa < wa1) te[base + (size_t)wa * HW + s.iy * a.W + s.ix] = narrow<TL>(1.0f);
        }
    }
}

template <typename TL>
cudaError_t encode_as(EncodeArgs a, int B, int sms, cudaStream_t st) {
    const int rows = a.E * a.sH * a.sW;
    const int HW = a.H * a.W, S = a.sH * a.sW;
    const size_t smem_small = ((size_t)a.K * HW + 15) & ~(size_t)15;
    if (a.sweep && rows > 0 && (HW & 3) == 0 && (a.W & 3) == 0 && (HW >> 2) <= 256 && (size_t)2 * HW <= 48 * 1024) {
        // vector shapes: the [K, H, W] grids by one small launch, the limb tensors by the address-ordered sweep
        EncodeArgs small = a;
        small.small_only = 1;
        if (smem_small > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(encode_targets_kernel<TL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_small);
            if (e != cudaSuccess) return e;
        }
        encode_targets_kernel<TL><<<dim3(B, 1), 256, smem_small, st>>>(small);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        // tiles of about 48 KB per tensor, whole rows
        int rows_per_tile = (48 * 1024) / (HW * (int)sizeof(TL));
        if (rows_per_tile < 1) rows_per_tile = 1;
        if (rows_per_tile > S) rows_per_tile = S;
        const int chunks = (S + rows_per_tile - 1) / rows_per_tile;
        rows_per_tile = (S + chunks - 1) / chunks;
        const long long n_tiles = (long long)B * a.E * chunks;
        const int grid = (int)std::min<long long>(n_tiles, (long long)sms * a.sweep_ctas_per_sm);
        encode_sweep_kernel<TL><<<grid, 256, (size_t)2 * HW, st>>>(a, B, chunks, rows_per_tile);
        return cudaGetLastError();
    }
    // enough CTAs to fill the machine a few times over; every CTA rebuilds the image's byte map (cheap)
    int Z = (4 * sms + B - 1) / B;
    if (Z < 1) Z = 1;
    if (Z > rows) Z = rows > 0 ? rows : 1;
    a.rows_per_cta = rows > 0 ? (rows + Z - 1) / Z : 0;
    Z = rows > 0 ? (rows + a.rows_per_cta - 1) / a.rows_per_cta : 1;
    const size_t smem = ((size_t)a.K * a.H * a.W + 15) & ~(size_t)15;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(encode_targets_kernel<TL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    encode_targets_kernel<TL><<<dim3(B, Z), 256, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_encode_targets(EncodeArgs a, int B, int sms, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    switch (a.limb_dtype) {
        case HEAD_F32: return encode_as<float>(a, B, sms, st);
        case HEAD_F16: return encode_as<__half>(a, B, sms, st);
        case HEAD_BF16: return encode_as<__nv_bfloat16>(a, B, sms, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace ppn
