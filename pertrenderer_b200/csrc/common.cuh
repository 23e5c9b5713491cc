// Shared device helpers of the perturbed shading kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/pertshade.h"

namespace pert {

constexpr int NT = 128;  // threads per CTA of the stand-alone operator kernels
constexpr int NW = NT / 32;
// The fused shader kernels run ONE WARP per CTA: tiles differ a lot in cost (sparse fragments), and a
// CTA only gives its shared memory back when its slowest warp is done; with one-warp CTAs the hardware
// CTA scheduler balances the load per tile.
constexpr int FNT = 32;
constexpr int FBT = 64;  // threads per CTA of the fallback pass: two independent warps
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ int warp_max_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ float warp_prod(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v *= __shfl_xor_sync(FULL, v, o);
    return v;
}
// (value, index) max with the FIRST index winning ties
__device__ __forceinline__ void warp_argmax(float& v, int& i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(FULL, v, o);
        const int oi = __shfl_xor_sync(FULL, i, o);
        if (ov > v || (ov == v && oi < i)) {
            v = ov;
            i = oi;
        }
    }
}

// ---- reductions over an aligned group of G lanes (G a power of two, warp-uniform; a compile-time
// constant in the production instantiations, so these loops unroll) -------------------------------
__device__ __forceinline__ float group_sum(float v, int G) {
#pragma unroll
    for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ int group_sum_i(int v, int G) {
#pragma unroll
    for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ int group_min_i(int v, int G) {
#pragma unroll
    for (int o = G >> 1; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ float group_prod(float v, int G) {
#pragma unroll
    for (int o = G >> 1; o > 0; o >>= 1) v *= __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ void group_argmax(float& v, int& i, int G) {
#pragma unroll
    for (int o = G >> 1; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(FULL, v, o);
        const int oi = __shfl_xor_sync(FULL, i, o);
        if (ov > v || (ov == v && oi < i)) {
            v = ov;
            i = oi;
        }
    }
}

__host__ __device__ __forceinline__ int pow2_ceil(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}
__host__ __device__ __forceinline__ int pow2_floor(int v) {
    int p = 1;
    while (p * 2 <= v) p <<= 1;
    return p;
}

// warp-aggregated append of `flag`-ed items to a shared work list (CTA-shared counter)
__device__ __forceinline__ void list_append(bool flag, uint16_t item, uint16_t* list, int* count) {
    const unsigned b = __ballot_sync(FULL, flag);
    if (b == 0) return;
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == __ffs(b) - 1) base = atomicAdd(count, __popc(b));
    base = __shfl_sync(FULL, base, __ffs(b) - 1);
    if (flag) list[base + __popc(b & ((1u << lane) - 1u))] = item;
}

// number of SMs of the current device (persistent grids are sized in multiples of it); cached per device
static inline int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// Grid of a persistent kernel: as many CTAs as the device holds at once (registers and shared memory decide)
template <class Kern>
static inline unsigned resident_grid(Kern kern, int threads, size_t smem) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, threads, smem) != cudaSuccess || nb < 1) nb = 1;
    return (unsigned)(sm_count() * nb);
}

// Shared-memory layout of a kernel: computed ONCE on the host (byte offsets in the launch record), so the
// kernels spend one add per array instead of re-deriving the layout (the fused kernels are instruction-fetch
// sensitive: every instruction of glue counts).
static inline size_t carve(size_t n, size_t sz) { return ((n * sz) + 15) & ~(size_t)15; }
constexpr int MAX_SMEM_ARRAYS = 20;
struct SmemLayout {
    int off[MAX_SMEM_ARRAYS];
    int n;
    int bytes;
};
struct Carver {  // host side
    SmemLayout& L;
    explicit Carver(SmemLayout& l) : L(l) { L.n = 0; L.bytes = 0; }
    void take(size_t count, size_t elem) {
        L.off[L.n++] = L.bytes;
        L.bytes += (int)((count * elem + 15) & ~(size_t)15);
    }
};
struct Taker {  // device side
    unsigned char* base;
    const SmemLayout& L;
    int i;
    __device__ Taker(unsigned char* b, const SmemLayout& l) : base(b), L(l), i(0) {}
    template <typename T>
    __device__ __forceinline__ T* take() {
        return reinterpret_cast<T*>(base + L.off[i++]);
    }
};

__device__ __forceinline__ void store_winner(void* winners, int win_bytes, int64_t idx, int v) {
    if (win_bytes == 1) reinterpret_cast<uint8_t*>(winners)[idx] = (uint8_t)v;
    else reinterpret_cast<uint16_t*>(winners)[idx] = (uint16_t)v;
}
__device__ __forceinline__ int load_winner(const void* winners, int win_bytes, int64_t idx) {
    return win_bytes == 1 ? (int)reinterpret_cast<const uint8_t*>(winners)[idx]
                          : (int)reinterpret_cast<const uint16_t*>(winners)[idx];
}

// Geometry of one launch of the fused kernels.  One WARP owns a tile of `tp` consecutive pixels
// (tp*K fragment entries are one contiguous run of every (P,K) tensor); G = 32/tp lanes work on each
// pixel of the tile in the per-pixel phases.
struct Launch {
    int tp;         // pixels per warp tile: 4, 8, 16 or 32
    int G;          // lanes per pixel = 32 / tp
    int gshift;     // log2(G)
    int64_t P;      // pixels in this call
    int64_t HW;     // pixels per batch element
    int64_t ntiles; // ceil(P / tp)
    int win_bytes;  // 1 or 2
    int sa_loc;     // local aggregation samples (s_agg_end - s_agg_begin)
    int sc;         // backward: samples per shared-memory chunk (multiple of 32)
    int nchunks;    // backward: ceil(sa_loc / sc)
    int lpe_r, lpe_r_shift;  // coverage sampling: lanes per entry = min(32, pow2_ceil(local quads))
    int lpe_a, lpe_a_shift;  // argmax sampling: lanes per pixel = min(32, pow2_ceil(local quads))
    int lpp, lpp_shift;      // backward: lanes per (pixel, logit) pair = min(8, pow2_floor(local quads))
    int cap;        // capacity (valid entries) of the tile's compact arrays: tp*K, or tp*K/2 in sparse-first mode
    int warp_smem;  // bytes of shared memory per warp
    int warp_smem_rast;  // ... of the coverage-sample launch of a split fallback pass (forward)
    SmemLayout sm;  // where each array lives
    int vec_ok;     // tile rows are 16-byte aligned in every (P,K) tensor
    float invK;     // 1/K for the entry -> pixel division
    // launch constants computed once on the host (IEEE fp32, the same values the kernels used to derive)
    float gal;      // gamma / alpha (smoothagg.py:201)
    float inv_sigma, invSg, inv_sr, invS;  // 1/sigma, 1/(S_agg gamma), 1/(S_rast sigma), 1/S_agg
    float inv_gamma;  // 1/gamma (SoftAgg, smoothagg.py:181)
    float t_compound; // coverage entries with |x|/sigma >= this are drawn by the compound sampler (tile.cuh)
    float t_bucket[2]; // ... and bucketed by expected flips: [t_compound, t_bucket[0]) many, [.., t_bucket[1]) some, rest rare
    bool lean;         // backward: the pair list takes over the counts array (shade_bwd.cu bwd_smem_layout)
};

// 16-byte asynchronous global -> shared copy (LDGSTS) and its completion wait
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// Out-of-line helpers for rarely taken or bulky paths (code size, see SmemLayout)
static __device__ __noinline__ float logf_exact(float x) { return logf(x); }
static __device__ __noinline__ int lower_bound_u16(const uint16_t* v, int lo, int hi, int target) {
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((int)v[mid] < target) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
// zero n floats (one warp); 128-bit stores when the run is 16-byte aligned and a multiple of 4 floats
static __device__ __noinline__ void zero_fill(float* dst, int n, bool vec_ok) {
    const int lane = threadIdx.x & 31;
    if (vec_ok && (n & 3) == 0) {
        float4* d4 = reinterpret_cast<float4*>(dst) + lane;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        int left = (n >> 2) - lane;  // float4 slots from this lane's first one to the end
#pragma unroll 1
        for (; left > 96; left -= 128, d4 += 128) {  // four stores per trip, no per-store bookkeeping
            d4[0] = z;
            d4[32] = z;
            d4[64] = z;
            d4[96] = z;
        }
        if (left > 0) d4[0] = z;
        if (left > 32) d4[32] = z;
        if (left > 64) d4[64] = z;
    } else {
#pragma unroll 1
        for (int i = lane; i < n; i += 32) dst[i] = 0.f;
    }
}

// floor(log2(32 / n)) for 1 <= n: lanes per item that keep a warp full (no integer division)
__device__ __forceinline__ int fill_shift(int n) { return n >= 32 ? 0 : (n <= 1 ? 5 : 5 - (32 - __clz(n - 1))); }

// Lanes per item (log2) for `n` items of `nq` sample quads each: a lane group of 2^k lanes shares one item
// (each lane takes nq/2^k quads, then a k-level shuffle reduction).  Picks the k <= kmax with the fewest
// issued instructions: passes * (quads per lane * cost of one quad + reduction).
__device__ __forceinline__ int best_lane_shift(int n, int nq, int kmax) {
    int best_k = 0, best_c = 0x7fffffff;
#pragma unroll 1
    for (int k = 0; k <= kmax; ++k) {
        const int passes = ((n << k) + 31) >> 5;
        const int per_lane = (nq + (1 << k) - 1) >> k;
        const int c = passes * (per_lane * 100 + 24 + 6 * k);
        if (c < best_c) {
            best_c = c;
            best_k = k;
        }
    }
    return best_k;
}

// batch element of pixel gp: pixels of a tile span at most two images, so one 32-bit division per tile
__device__ __forceinline__ int batch_of(int64_t pix0, int p, int64_t HW) {
    const unsigned hw = (unsigned)HW;
    const unsigned b0 = (unsigned)pix0 / hw;  // P < 2^31 (checked by the C ABI)
    unsigned r = (unsigned)pix0 - b0 * hw + (unsigned)p;
    unsigned b = b0;
    while (r >= hw) {  // tiny images: a tile may cover several
        r -= hw;
        b++;
    }
    return (int)b;
}

// Tile blob (optional saved state of the sparse-first main pass): what backward would otherwise recompute
// from pix_to_face / zbuf / counts -- the compact valid list and the per-pixel logit summary of forward.
// 32-bit words per tile:  [0] nv (-1: the tile went to the fallback pass)   [1 .. tp+1] vstart[0..tp]
//   then 6 per pixel: zmax, zimax, prod_nz, zeta_max, argzi | a0 << 16, nzero | kpad << 16
//   then vlist (u16 x cap), cnt (u16 x cap), zeta (f32 x cap)
__host__ __device__ __forceinline__ int blob_words(int tp, int cap) { return ((2 + 7 * tp + 2 * cap) + 3) & ~3; }
__host__ __device__ __forceinline__ int blob_pix_off(int tp) { return 2 + tp; }
__host__ __device__ __forceinline__ int blob_vlist_off(int tp) { return 2 + 7 * tp; }
__host__ __device__ __forceinline__ int blob_cnt_off(int tp, int cap) { return 2 + 7 * tp + cap / 2; }
__host__ __device__ __forceinline__ int blob_zeta_off(int tp, int cap) { return 2 + 7 * tp + cap; }

// entry index within a tile -> pixel of the tile.  Exact for e < 2^16, K < 2^10: (e + .5)/K is at
// least .5/K away from an integer, far more than the fp32 rounding of the product.
__device__ __forceinline__ int entry_pixel(int e, float invK) { return __float2int_rz(((float)e + 0.5f) * invK); }

}  // namespace pert
