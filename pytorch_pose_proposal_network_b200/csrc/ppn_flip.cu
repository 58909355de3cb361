// The flip test's merge (ppn_flip_merge): average a head with the mirrored head of its horizontally flipped input.
// The rule is specified in DESIGN.md §15.
//
// One pass, bandwidth-bound: A (the head) and Bf (the flipped view's head) are read once, `out` written once.  A CTA
// takes a chunk of consecutive output planes (global plane index b * C + c), as many as fit 1024 access units of
// 16 bytes (vector path) or one element (scalar path):
//   1. the source plane of each output plane of the chunk is looked up once, from the part and limb mirror tables
//      that travel in the kernel parameters (no device table, no copies);
//   2. the source planes are staged in shared memory with coalesced loads while each thread loads its own units of A;
//   3. each thread composes its output units from its A values and the staged planes read with their columns
//      reversed.  Rows of 12 fp16 / bf16 cells are not a multiple of 16 bytes, so a unit can straddle rows and the
//      reversal is not a lane swizzle inside one vector; reading the staged plane element by element handles every W.
//      16-bit heads with an even W read the staged plane a 32-bit pair of mirrored cells at a time.
// The vector path needs 16-byte aligned heads and planes of a multiple of 16 bytes (every preset's grid in every
// dtype).  Other shapes (odd grids such as 13 x 13, a 1 x 1 grid) and heads that are only element-aligned take the
// scalar path: the same kernel with one-element units.  `out` may be `head` (each unit of A is read by the thread that
// writes it); it never overlaps Bf (the C ABI rejects that).
#include "ppn_kernels.h"

namespace ppn {

namespace {

constexpr int kFlipThreads = 256;
constexpr int kFlipItems = 4;                                  // units per thread per chunk
constexpr int kFlipUnits = kFlipThreads * kFlipItems;          // 1024 units: 16 KB of staged Bf on the vector path
constexpr uint32_t kXBit = 0x80000000u;                        // source-table flag: an x-group plane

template <typename T, int N>
struct alignas(sizeof(T) * N) Unit { T v[N]; };

template <typename T> __device__ __forceinline__ T from_bits(uint16_t b);
template <> __device__ __forceinline__ __half from_bits<__half>(uint16_t b) { return __ushort_as_half(b); }
template <> __device__ __forceinline__ __nv_bfloat16 from_bits<__nv_bfloat16>(uint16_t b) { return __ushort_as_bfloat16(b); }

template <typename T, int N>
__global__ void __launch_bounds__(kFlipThreads) flip_merge_kernel(const FlipMergeArgs a) {
    using U = Unit<T, N>;
    __shared__ __align__(16) unsigned char stage_raw[kFlipUnits * sizeof(U)];
    __shared__ uint32_t src_of[kFlipUnits];                    // per chunk plane: source plane index | kXBit
    U* stage = reinterpret_cast<U*>(stage_raw);
    const T* staged = reinterpret_cast<const T*>(stage_raw);

    const int tid = threadIdx.x;
    const int vpp = a.HW / N;                                  // units per plane
    const uint32_t first = blockIdx.x * (uint32_t)a.chunk_planes;
    const int np = (int)min((uint32_t)a.chunk_planes, a.planes - first);
    const int nu = np * vpp;

    const int K = a.K, C = a.C, parts = 6 * a.K;
    for (int l = tid; l < np; l += kFlipThreads) {
        const uint32_t gp = first + l;
        const uint32_t b = gp / (uint32_t)C;
        const int c = (int)(gp - b * (uint32_t)C);
        int s;
        uint32_t x = 0;
        if (c < parts) {
            const int g = c / K, k = c - g * K;
            s = g * K + a.part_mirror[k];
            x = g == 2 ? kXBit : 0u;
        } else {
            const int r = (c - parts) / a.sW, col = (c - parts) - r * a.sW;   // r = e * sH + row of the window
            const int e = r / a.sH, row = r - e * a.sH;
            s = parts + (a.limb_mirror[e] * a.sH + row) * a.sW + (a.sW - 1 - col);
        }
        src_of[l] = (b * (uint32_t)C + (uint32_t)s) | x;
    }
    __syncthreads();

    const U* __restrict__ flipped = reinterpret_cast<const U*>(a.flipped);
    const U* head = reinterpret_cast<const U*>(a.head) + (size_t)first * vpp;
    U* out = reinterpret_cast<U*>(a.out) + (size_t)first * vpp;
    U fv[kFlipItems], av[kFlipItems];
#pragma unroll
    for (int it = 0; it < kFlipItems; ++it) {
        const int u = tid + it * kFlipThreads;
        if (u < nu) {
            const int l = u / vpp;
            fv[it] = flipped[(size_t)(src_of[l] & ~kXBit) * vpp + (u - l * vpp)];
            av[it] = head[u];
        }
    }
#pragma unroll
    for (int it = 0; it < kFlipItems; ++it) {
        const int u = tid + it * kFlipThreads;
        if (u < nu) stage[u] = fv[it];
    }
    __syncthreads();

    const int W = a.W;
#pragma unroll
    for (int it = 0; it < kFlipItems; ++it) {
        const int u = tid + it * kFlipThreads;
        if (u >= nu) continue;
        const int l = u / vpp;
        const bool is_x = (src_of[l] & kXBit) != 0;
        const int cell = (u - l * vpp) * N;
        const int i = cell / W;
        int j = cell - i * W;
        int s = l * a.HW + i * W + (W - 1 - j);                // staged element of the mirrored cell
        U o;
        if constexpr (sizeof(T) == 2 && N > 1) {
            if ((W & 1) == 0) {
                // Even W: cells (j, j + 1), j even, mirror to the staged pair (s, s - 1), s odd, which is one aligned
                // 32-bit word with s in its high half.  Half the shared-memory reads of the element loop.
                const uint32_t* staged32 = reinterpret_cast<const uint32_t*>(stage_raw);
#pragma unroll
                for (int k = 0; k < N; k += 2) {
                    const uint32_t w = staged32[(s - 1) >> 1];
                    float hi = widen(from_bits<T>((uint16_t)(w >> 16))), lo = widen(from_bits<T>((uint16_t)(w & 0xffffu)));
                    if (is_x) { hi = __fsub_rn(1.0f, hi); lo = __fsub_rn(1.0f, lo); }
                    o.v[k] = narrow<T>(__fmul_rn(__fadd_rn(widen(av[it].v[k]), hi), 0.5f));
                    o.v[k + 1] = narrow<T>(__fmul_rn(__fadd_rn(widen(av[it].v[k + 1]), lo), 0.5f));
                    if ((j += 2) == W) { j = 0; s += 2 * W - 2; }   // next row: its last two columns
                    else s -= 2;
                }
                out[u] = o;
                continue;
            }
        }
#pragma unroll
        for (int k = 0; k < N; ++k) {
            float bv = widen(staged[s]);
            if (is_x) bv = __fsub_rn(1.0f, bv);
            o.v[k] = narrow<T>(__fmul_rn(__fadd_rn(widen(av[it].v[k]), bv), 0.5f));
            if (++j == W) { j = 0; s += 2 * W - 1; }           // next row: its last column
            else --s;
        }
        out[u] = o;
    }
}

template <typename T>
cudaError_t launch_t(const FlipMergeArgs& a, cudaStream_t st) {
    constexpr int N = 16 / sizeof(T);
    const int unit = a.vec ? N : 1;
    FlipMergeArgs b = a;
    b.chunk_planes = kFlipUnits / (a.HW / unit);
    const unsigned grid = (unsigned)((a.planes + b.chunk_planes - 1) / b.chunk_planes);
    if (a.vec) flip_merge_kernel<T, N><<<grid, kFlipThreads, 0, st>>>(b);
    else flip_merge_kernel<T, 1><<<grid, kFlipThreads, 0, st>>>(b);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_flip_merge(const FlipMergeArgs& a, int dtype, cudaStream_t st) {
    if (dtype == HEAD_F16) return launch_t<__half>(a, st);
    if (dtype == HEAD_BF16) return launch_t<__nv_bfloat16>(a, st);
    return launch_t<float>(a, st);
}

}  // namespace ppn
