// Batch augmentation (ppn_augment_images, ppn_augment_people): warp, flip and normalise a ragged uint8 image batch,
// and move its annotations with it.  The rule is specified in DESIGN.md §14.
//
// Images.  One CTA per (output tile, image), one launch for the batch.  A thread computes P = 16 / sizeof(OutT)
// consecutive output pixels of one row, three channels each: 3 * P values, stored as three 16-byte vectors in either
// layout.  Before computing, the CTA maps the four corner pixels of its tile through M; the bounding box of their
// taps, widened by one pixel, is the tile's source footprint.  When the footprint fits the staging budget and holds
// at most two source pixels per output pixel, it is copied to shared memory in aligned 16-byte words (coalesced,
// whatever the byte alignment of the rows); taps that fall outside it anyway (rounding at the tile's border) read
// global memory.  Otherwise (minification) every tap is gathered through L1.  Either way a tap reads the same byte,
// so staging never changes a result.
//
// People.  One thread per person: keypoints and box corners through A in fp64, the box as the bounds of its four
// corners, part columns permuted left <-> right on a flipped image, the part size scaled by sqrt|det A|.
#include "ppn_kernels.h"

namespace ppn {

namespace {

constexpr int kAugThreads = 256;
constexpr int kTileW = 64;                           // output tile width: 16 (fp32) or 8 (16-bit) threads per row
constexpr float kCoordLimit = 1073741824.0f;         // 2^30: beyond it (or non-finite) a coordinate reads the fill

// source coordinate of output pixel (u, v): ((m0 * pcx + m1 * pcy) + m2) - 0.5, one rounding per operation
__device__ __forceinline__ float src_coord(float m0, float m1, float m2, float pcx, float pcy) {
    return __fsub_rn(__fadd_rn(__fadd_rn(__fmul_rn(m0, pcx), __fmul_rn(m1, pcy)), m2), 0.5f);
}

__device__ __forceinline__ bool coord_ok(float s) { return fabsf(s) <= kCoordLimit; }   // false for NaN and +-inf

template <typename OutT> struct Words;               // 3 * P output values as twelve 32-bit words, lower address first
template <> struct Words<float> {
    static __device__ __forceinline__ uint32_t at(const float* v, int i) { return __float_as_uint(v[i]); }
};
template <> struct Words<__half> {
    static __device__ __forceinline__ uint32_t at(const float* v, int i) { return pack2<__half>(v[2 * i], v[2 * i + 1]); }
};
template <> struct Words<__nv_bfloat16> {
    static __device__ __forceinline__ uint32_t at(const float* v, int i) {
        return pack2<__nv_bfloat16>(v[2 * i], v[2 * i + 1]);
    }
};

template <typename OutT>
__device__ __forceinline__ void store_vec(OutT* dst, const float* v /* [P] per vector, 4 / 8 / 12 words */, int n_vec) {
    uint4* d = reinterpret_cast<uint4*>(dst);
#pragma unroll
    for (int k = 0; k < 3; ++k)
        if (k < n_vec)
            d[k] = make_uint4(Words<OutT>::at(v, 4 * k), Words<OutT>::at(v, 4 * k + 1), Words<OutT>::at(v, 4 * k + 2),
                              Words<OutT>::at(v, 4 * k + 3));
}

template <typename OutT, bool kNHWC>
__global__ void __launch_bounds__(kAugThreads) augment_images_kernel(const AugmentArgs a) {
    constexpr int P = 16 / (int)sizeof(OutT);
    constexpr int kRowThreads = kTileW / P;
    constexpr int kTileH = kAugThreads / kRowThreads;
    extern __shared__ __align__(16) uint8_t stage[];

    const int b = blockIdx.z;
    const int x0 = blockIdx.x * kTileW, y0 = blockIdx.y * kTileH;
    const float* Mb = a.M + 6 * (size_t)b;
    const float m00 = __ldg(Mb), m01 = __ldg(Mb + 1), m02 = __ldg(Mb + 2);
    const float m10 = __ldg(Mb + 3), m11 = __ldg(Mb + 4), m12 = __ldg(Mb + 5);
    const int h = __ldg(a.hw + 2 * b), w = __ldg(a.hw + 2 * b + 1);
    const uint8_t* img = a.pixels + __ldg(a.offset + b);

    // ---- the tile's source footprint (CTA-uniform) ----
    int fx0 = 0, fx1 = -1, fy0 = 0, fy1 = -1, pitch = 0;
    bool staged = false;
    if (a.stage_bytes > 0) {
        const float cu[2] = {x0 + 0.5f, min(x0 + kTileW, a.outW) - 0.5f};
        const float cv[2] = {y0 + 0.5f, min(y0 + kTileH, a.outH) - 0.5f};
        float lx = 0.f, hx = 0.f, ly = 0.f, hy = 0.f;
        bool ok = true;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float sx = src_coord(m00, m01, m02, cu[i & 1], cv[i >> 1]);
            const float sy = src_coord(m10, m11, m12, cu[i & 1], cv[i >> 1]);
            ok = ok && coord_ok(sx) && coord_ok(sy);
            lx = i ? fminf(lx, sx) : sx; hx = i ? fmaxf(hx, sx) : sx;
            ly = i ? fminf(ly, sy) : sy; hy = i ? fmaxf(hy, sy) : sy;
        }
        if (ok) {
            fx0 = max((int)floorf(lx) - 1, 0); fx1 = min((int)floorf(hx) + 2, w - 1);
            fy0 = max((int)floorf(ly) - 1, 0); fy1 = min((int)floorf(hy) + 2, h - 1);
            if (fx0 <= fx1 && fy0 <= fy1) {
                pitch = (3 * (fx1 - fx0 + 1) + 30) >> 4;          // 16-byte words per staged row, any start phase
                // staged only where the taps are dense: a minifying footprint holds rows and columns no tap reads,
                // which the L1 gather never fetches (measured, DESIGN.md §14)
                staged = (long long)(fy1 - fy0 + 1) * pitch * 16 <= a.stage_bytes &&
                         (fy1 - fy0 + 1) * (fx1 - fx0 + 1) <= 2 * kTileW * kTileH;
            }
        }
    }
    if (staged) {
        const int rows = fy1 - fy0 + 1, nb = 3 * (fx1 - fx0 + 1);
        for (int i = threadIdx.x; i < rows * pitch; i += kAugThreads) {
            const int r = i / pitch, k = i - r * pitch;
            const uintptr_t row = reinterpret_cast<uintptr_t>(img + ((long long)(fy0 + r) * w + fx0) * 3);
            const uintptr_t first = row & ~(uintptr_t)15;
            // only words holding a byte of the row: they lie inside the buffer's 16-byte granules
            if (first + 16 * (uintptr_t)k < row + nb)
                reinterpret_cast<uint4*>(stage)[i] = __ldg(reinterpret_cast<const uint4*>(first) + k);
        }
        __syncthreads();
    }

    const int tx = threadIdx.x % kRowThreads, ty = threadIdx.x / kRowThreads;
    const int v = y0 + ty, u0 = x0 + tx * P;
    if (v >= a.outH || u0 >= a.outW) return;

    auto tap = [&](int x, int y, float* p) {
        if (x < 0 || x >= w || y < 0 || y >= h) {
            p[0] = a.fill[0]; p[1] = a.fill[1]; p[2] = a.fill[2];
            return;
        }
        const uint8_t* s;
        if (staged && x >= fx0 && x <= fx1 && y >= fy0 && y <= fy1) {
            const uintptr_t row = reinterpret_cast<uintptr_t>(img + ((long long)y * w + fx0) * 3);
            s = stage + (y - fy0) * pitch * 16 + (int)(row & 15) + 3 * (x - fx0);
            p[0] = s[0]; p[1] = s[1]; p[2] = s[2];
        } else {
            s = img + ((long long)y * w + x) * 3;
            p[0] = __ldg(s); p[1] = __ldg(s + 1); p[2] = __ldg(s + 2);
        }
    };

    float val[3 * P];                                 // NCHW: [c][j]   NHWC: [j][c]
    const float pcy = v + 0.5f;
#pragma unroll
    for (int j = 0; j < P; ++j) {
        const float pcx = (u0 + j) + 0.5f;
        const float sx = src_coord(m00, m01, m02, pcx, pcy), sy = src_coord(m10, m11, m12, pcx, pcy);
        float r[3] = {a.fill[0], a.fill[1], a.fill[2]};
        if (coord_ok(sx) && coord_ok(sy)) {
            const float fx = floorf(sx), fy = floorf(sy);
            const int ix = (int)fx, iy = (int)fy;
            if (ix + 1 >= 0 && ix < w && iy + 1 >= 0 && iy < h) {        // some tap inside the source
                const float ax = __fsub_rn(sx, fx), ay = __fsub_rn(sy, fy);
                const float bx = __fsub_rn(1.0f, ax), by = __fsub_rn(1.0f, ay);
                float p00[3], p01[3], p10[3], p11[3];
                tap(ix, iy, p00); tap(ix + 1, iy, p01); tap(ix, iy + 1, p10); tap(ix + 1, iy + 1, p11);
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float top = __fadd_rn(__fmul_rn(p00[c], bx), __fmul_rn(p01[c], ax));
                    const float bot = __fadd_rn(__fmul_rn(p10[c], bx), __fmul_rn(p11[c], ax));
                    r[c] = __fadd_rn(__fmul_rn(top, by), __fmul_rn(bot, ay));
                }
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float o = __fdiv_rn(__fsub_rn(__fmul_rn(r[c], a.in_scale), a.mean[c]), a.std[c]);
            val[kNHWC ? 3 * j + c : c * P + j] = o;
        }
    }

    OutT* out = static_cast<OutT*>(a.out);
    const int n_px = min(P, a.outW - u0);
    if (kNHWC) {
        OutT* dst = out + (((size_t)b * a.outH + v) * a.outW + u0) * 3;
        if (a.vec && n_px == P) {
            store_vec<OutT>(dst, val, 3);
        } else {
#pragma unroll
            for (int i = 0; i < 3 * P; ++i)
                if (i < 3 * n_px) dst[i] = narrow<OutT>(val[i]);
        }
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            OutT* dst = out + (((size_t)b * 3 + c) * a.outH + v) * a.outW + u0;
            if (a.vec && n_px == P) {
                store_vec<OutT>(dst, val + c * P, P * (int)sizeof(OutT) / 16);
            } else {
#pragma unroll
                for (int j = 0; j < P; ++j)
                    if (j < n_px) dst[j] = narrow<OutT>(val[c * P + j]);
            }
        }
    }
}

// first image b with person_off[b + 1] > p, clamped to [0, B - 1] (a malformed table cannot index outside A)
__device__ __forceinline__ int image_of(const int32_t* off, int B, int p) {
    int lo = 0, hi = B - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(off + mid + 1) > p) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__device__ __forceinline__ double affine(double c0, double c1, double c2, double x, double y) {
    return __dadd_rn(__dadd_rn(__dmul_rn(c0, x), __dmul_rn(c1, y)), c2);
}

__global__ void __launch_bounds__(kAugThreads) augment_people_kernel(const AugmentPeopleArgs a) {
    const int p = blockIdx.x * kAugThreads + threadIdx.x;
    if (p >= a.n) return;
    const int b = image_of(a.person_off, a.B, p);
    const double* A = a.A + 6 * (size_t)b;
    const double a00 = A[0], a01 = A[1], a02 = A[2], a10 = A[3], a11 = A[4], a12 = A[5];
    const bool flip = a.flip[b] != 0;
    const int J = a.J;
    for (int i = 0; i < J; ++i) {
        const int s = flip ? a.perm[i] : i;
        const size_t src = (size_t)p * J + s, dst = (size_t)p * J + i;
        const double x = a.keypoints[2 * src], y = a.keypoints[2 * src + 1];
        a.keypoints_out[2 * dst] = __double2float_rn(affine(a00, a01, a02, x, y));
        a.keypoints_out[2 * dst + 1] = __double2float_rn(affine(a10, a11, a12, x, y));
        a.visible_out[dst] = a.visible[src];
    }
    const double cx = a.bbox[4 * p], cy = a.bbox[4 * p + 1], bw = a.bbox[4 * p + 2], bh = a.bbox[4 * p + 3];
    double* bo = a.bbox_out + 4 * (size_t)p;
    if (bw > 0 && bh > 0) {
        const double hw = __dmul_rn(bw, 0.5), hh = __dmul_rn(bh, 0.5);
        const double xs[2] = {__dsub_rn(cx, hw), __dadd_rn(cx, hw)}, ys[2] = {__dsub_rn(cy, hh), __dadd_rn(cy, hh)};
        double lx = 0, hx = 0, ly = 0, hy = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {                 // corners (x-, y-), (x+, y-), (x-, y+), (x+, y+)
            const double X = affine(a00, a01, a02, xs[i & 1], ys[i >> 1]);
            const double Y = affine(a10, a11, a12, xs[i & 1], ys[i >> 1]);
            lx = (i == 0 || X < lx) ? X : lx; hx = (i == 0 || X > hx) ? X : hx;
            ly = (i == 0 || Y < ly) ? Y : ly; hy = (i == 0 || Y > hy) ? Y : hy;
        }
        bo[0] = __dmul_rn(__dadd_rn(lx, hx), 0.5); bo[1] = __dmul_rn(__dadd_rn(ly, hy), 0.5);
        bo[2] = __dsub_rn(hx, lx); bo[3] = __dsub_rn(hy, ly);
    } else {                                          // unlabelled box: the centre moves, the box stays empty
        bo[0] = affine(a00, a01, a02, cx, cy); bo[1] = affine(a10, a11, a12, cx, cy);
        bo[2] = 0.0; bo[3] = 0.0;
    }
    a.size_out[p] = __dmul_rn(a.size[p], __dsqrt_rn(fabs(__dsub_rn(__dmul_rn(a00, a11), __dmul_rn(a01, a10)))));
}

template <typename OutT, bool kNHWC>
cudaError_t launch_images_t(const AugmentArgs& a, cudaStream_t st) {
    constexpr int P = 16 / (int)sizeof(OutT);
    constexpr int kTileH = kAugThreads / (kTileW / P);
    const dim3 grid((a.outW + kTileW - 1) / kTileW, (a.outH + kTileH - 1) / kTileH, a.B);
    augment_images_kernel<OutT, kNHWC><<<grid, kAugThreads, a.stage_bytes, st>>>(a);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_augment_images(const AugmentArgs& a, int out_dtype, bool nhwc, cudaStream_t st) {
    if (out_dtype == HEAD_F16) return nhwc ? launch_images_t<__half, true>(a, st) : launch_images_t<__half, false>(a, st);
    if (out_dtype == HEAD_BF16)
        return nhwc ? launch_images_t<__nv_bfloat16, true>(a, st) : launch_images_t<__nv_bfloat16, false>(a, st);
    return nhwc ? launch_images_t<float, true>(a, st) : launch_images_t<float, false>(a, st);
}

cudaError_t launch_augment_people(const AugmentPeopleArgs& a, cudaStream_t st) {
    augment_people_kernel<<<(a.n + kAugThreads - 1) / kAugThreads, kAugThreads, 0, st>>>(a);
    return cudaGetLastError();
}

}  // namespace ppn
