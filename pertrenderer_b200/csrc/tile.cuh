// Per-warp tile machinery shared by the fused forward and backward kernels.
//
// A warp owns `tp` consecutive pixels.  Real fragments are sparse in K (a handful of valid faces per
// pixel, padding last), so the tile is first reduced to a COMPACT list of its valid entries
// (pix_to_face >= 0); zbuf / dists / saved state are then touched only for those, and every later
// phase runs over compact indices n in [0, nv).  Reference semantics being reproduced:
//   random_rasterizer.py:46-48  mask, P = p_hat*mask, alpha = prod(1-P)
//   smoothagg.py:198-202        zi, zmax, zeta_k = (gamma/alpha) log P_k + zi_k - zmax, zeta_K = eps - zmax
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace pert {

// ------------------------------------------------------------------------------------------------
// phase 0: scan pix_to_face of the tile (128-bit loads), build the ascending list of valid entries
// ------------------------------------------------------------------------------------------------
// Returns the number of valid entries; only the first `cap` of them are written to vlist (a tile with
// more is handed to the fallback pass by the caller).
__device__ __forceinline__ int scan_valid(const int64_t* __restrict__ p2f /* tile base */, int E, bool vec_ok,
                                          uint16_t* vlist, int cap) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    int total = 0;
    constexpr int U = 4;  // loads in flight per lane
    for (int base = 0; base < E; base += 64 * U) {
        long long a[U], b[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e0 = base + u * 64 + 2 * lane;
            a[u] = -1;
            b[u] = -1;
            if (e0 + 1 < E) {
                if (vec_ok) {
                    const longlong2 v = __ldg(reinterpret_cast<const longlong2*>(p2f + e0));
                    a[u] = v.x;
                    b[u] = v.y;
                } else {
                    a[u] = __ldg(p2f + e0);
                    b[u] = __ldg(p2f + e0 + 1);
                }
            } else if (e0 < E) {
                a[u] = __ldg(p2f + e0);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (base + u * 64 >= E) break;  // warp-uniform
            const int e0 = base + u * 64 + 2 * lane;
            const bool v0 = a[u] >= 0, v1 = b[u] >= 0;
            const unsigned be = __ballot_sync(FULL, v0), bo = __ballot_sync(FULL, v1);
            const int pos = total + __popc(be & lt) + __popc(bo & lt);
            if (v0 && pos < cap) vlist[pos] = (uint16_t)e0;
            if (v1 && pos + (v0 ? 1 : 0) < cap) vlist[pos + (v0 ? 1 : 0)] = (uint16_t)(e0 + 1);
            total += __popc(be) + __popc(bo);
        }
    }
    return total;
}

// vstart[p] = first compact index of pixel p (p = 0..tp), by binary search on the ascending vlist
__device__ __forceinline__ void pixel_ranges(const uint16_t* vlist, int nv, int K, int tp, int* vstart) {
    const int lane = threadIdx.x & 31;
#pragma unroll 1
    for (int p = lane; p <= tp; p += 32) {
        vstart[p] = lower_bound_u16(vlist, 0, nv, p * K);
    }
}

// ------------------------------------------------------------------------------------------------
// stage 1: coverage samples of the listed entries
//   randomras/smoothrast.py:32-36: h = 1[x + sigma*U >= 0] (rounded multiply, rounded add), mean over s
//   saved for backward: cnt = sum_s h, rs = sum_s (h - h0) psi(U)   (smoothrast.py:46,49; psi = noise_score<SCORE>)
//   WOVR = true, without the control variate (randomHeaviside_wovr, smoothrast.py:61-108): rs = sum_s h psi(U); the
//   radius gate then only applies to x < 0 (h0 = 0), where a sample that cannot flip adds nothing
//   RENDER = true (forward-only render): counts only, rs is neither accumulated nor written; the same draws and h tests
// rlist holds compact indices n; xs/cnt/rs are compact arrays.
// ------------------------------------------------------------------------------------------------
template <class NoiseT, int SCORE = 0, bool WOVR = false, bool RENDER = false>
__device__ __forceinline__ void rast_sample_list(const NoiseT& noise, const uint16_t* rlist, int nlist,
                                                 const uint16_t* vlist, const float* xs, uint16_t* cnt, float* rs,
                                                 int K, float invK, int64_t pix0, float sigma, float inv_sigma,
                                                 int s_begin, int s_end, bool gate_ok,
                                                 int lpe_max /* lanes per entry at most */) {
    const int lane = threadIdx.x & 31;
    const int qb = s_begin >> 2, qe = (s_end + 3) >> 2;
    if (nlist == 0) return;
    // lanes per entry: as many as keep the warp full (few listed entries -> split an entry's samples over
    // more lanes; many -> one lane walks all the quads of its entry and no cross-lane reduction is needed)
    const int lpe_shift = min(31 - __clz(lpe_max), fill_shift(nlist));
    const int lpe = 1 << lpe_shift;
    const int gpw = 32 >> lpe_shift;  // entries per warp pass
    const int lig = lane & (lpe - 1);
#pragma unroll 1
    for (int base = 0; base < nlist; base += gpw) {
        const int li = base + (lane >> lpe_shift);
        const bool active = li < nlist;
        const int n = active ? rlist[li] : 0;
        const int e = vlist[n];
        const int pix = entry_pixel(e, invK), k = e - pix * K;
        const float x = xs[n];
        const bool h0 = x >= 0.0f;
        int c = 0;
        float r = 0.0f;
        if (active) {
            if constexpr (NoiseT::kBounded) {
                // a pair of samples can only flip when its Box-Muller radius reaches |x|/sigma: decide that
                // on the raw word and skip the transcendental work otherwise (exact, see radius_gate)
                const uint32_t gate = (gate_ok && !(WOVR && h0)) ? radius_gate(fabsf(x) * inv_sigma * 0.99999f) : 0u;
#pragma unroll 1
                for (int q = qb + lig; q < qe; q += lpe) {
                    uint32_t w[4];
                    noise.words(q, k, pix0 + pix, w);
#pragma unroll
                    for (int hp = 0; hp < 2; ++hp) {
                        const int s0 = q * 4 + hp * 2;
                        const bool in0 = s0 >= s_begin && s0 < s_end, in1 = s0 + 1 >= s_begin && s0 + 1 < s_end;
                        if ((w[hp * 2] >> 9) < gate) {
                            if (h0) c += (in0 ? 1 : 0) + (in1 ? 1 : 0);
                        } else {
                            float n0, n1;
                            box_muller(w[hp * 2], w[hp * 2 + 1], n0, n1);
                            const bool ha = __fadd_rn(x, __fmul_rn(sigma, n0)) >= 0.0f;
                            const bool hb = __fadd_rn(x, __fmul_rn(sigma, n1)) >= 0.0f;
                            if constexpr (RENDER) {
                                c += (in0 && ha ? 1 : 0) + (in1 && hb ? 1 : 0);
                            } else if constexpr (WOVR) {
                                if (in0) {
                                    c += ha ? 1 : 0;
                                    if (ha) r += n0;
                                }
                                if (in1) {
                                    c += hb ? 1 : 0;
                                    if (hb) r += n1;
                                }
                            } else {
                                if (in0) {
                                    c += ha ? 1 : 0;
                                    if (ha != h0) r += ha ? n0 : -n0;
                                }
                                if (in1) {
                                    c += hb ? 1 : 0;
                                    if (hb != h0) r += hb ? n1 : -n1;
                                }
                            }
                        }
                    }
                }
            } else {
#pragma unroll 1
                for (int q = qb + lig; q < qe; q += lpe) {
                    float nz[4];
                    noise.get4(q, k, pix0 + pix, nz);
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const int s = q * 4 + t;
                        const bool h = __fadd_rn(x, __fmul_rn(sigma, nz[t])) >= 0.0f;
                        if (s >= s_begin && s < s_end) {
                            c += h ? 1 : 0;
                            if constexpr (RENDER) {
                            } else if constexpr (WOVR) {
                                if (h) r += noise_score<SCORE>(nz[t]);
                            } else if (h != h0) {
                                r += h ? noise_score<SCORE>(nz[t]) : -noise_score<SCORE>(nz[t]);
                            }
                        }
                    }
                }
            }
        }
#pragma unroll 1
        for (int o = lpe >> 1; o > 0; o >>= 1) {
            c += __shfl_xor_sync(FULL, c, o);
            if constexpr (!RENDER) r += __shfl_xor_sync(FULL, r, o);
        }
        if (active && lig == 0) {
            cnt[n] = (uint16_t)c;
            if constexpr (!RENDER) rs[n] = r;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// stage 1, compound sampler (the default with in-kernel noise).  The pair (cnt, rs) of an entry depends on
// its samples only through the FLIPPED ones (h != h0).  Their number is F ~ Binomial(n, p) with
// p = Phi(-t), t = |x| / sigma, and given F each flipped sample contributes (h - h0) U = T, a standard normal
// conditioned on T > t (x >= 0: flips have U < -t and h - h0 = -1; x < 0: U >= t and h - h0 = +1).  So
//     cnt = h0 ? n - F : F,      rs = T_1 + ... + T_F
// drawn with ONE uniform for F (inversion on the survival function) and one per flip (inverse CDF of the
// tail) has exactly the joint law of the n per-sample draws of randomras/smoothrast.py:32-36,46, at a cost of
// O(1 + n p) instead of n normals: p = 0.02 two sigma inside a face.  Entries are independent of each other
// and of the aggregation noise, so every output of the shader keeps the law of the reference estimator; it is
// not the sample path of pert_noise_fill's tensor (PERT_F_PER_SAMPLE_NOISE restores that).
// Counters: (0x40000000 + 2*(s_begin/4) + call, k, pixel, stage 0): disjoint from every sample quad's and,
// for sample shards, from every other shard's (a shard of nq quads makes at most nq + 1 calls).
// ------------------------------------------------------------------------------------------------
template <class NoiseT>
struct CompoundCtx {
    NoiseT noise;
    const uint16_t* vlist;
    const float* xs;
    uint16_t* cnt;
    float* rs;
    int K;
    float invK;
    int64_t pix0;
    float inv_sigma;
    int n_loc;    // local coverage samples
    uint32_t c0;  // first counter
};

// The number of flips F of entry n (compound_entry): one uniform, the first word of counter c0.  Also returns what the
// tail draws need: the word quad of c0, p = Phi(-t) and t.
template <class NoiseT>
__device__ __forceinline__ int compound_flips(const CompoundCtx<NoiseT>& c, int k, int pix, float x, uint32_t (&w)[4],
                                              float& p, float& t) {
    t = fabsf(x) * c.inv_sigma;
    p = 0.5f * erfcf(t * 0.70710678118654752f);
    const float fn = (float)c.n_loc;
    const float nl = fn * log1pf(-p);
    const float sf1 = -expm1f(nl);  // P(F >= 1)
    c.noise.words(c.c0, (uint32_t)k, c.pix0 + pix, w);
    const float u = ((float)w[0] + 1.0f) * 2.3283064365386963e-10f;  // (0, 1], 2^-32 resolution near 0
    int F = 0;
    if (u <= sf1) {
        float pmf = __expf(nl), sf = sf1;
        const float ratio = __fdividef(p, 1.0f - p);
        // F >= k+1  <=>  u <= sf_k;  past the mode, stop once the terms are below the resolution of the running
        // difference (an event of probability < 1e-6 whose F is then off by a few)
        do {
            ++F;
            pmf *= ratio * __fdividef((float)(c.n_loc - F + 1), (float)F);
            sf -= pmf;
        } while (u <= sf && F < c.n_loc && (pmf > 1e-10f || (float)F < fn * p));
    }
    return F;
}

// one entry (compact index n) per calling lane; out of line: the body is bulky (erfc, log1p, expm1, erfcinv) and the
// fused kernels are instruction-fetch sensitive
template <class NoiseT>
static __device__ __noinline__ void compound_entry(const CompoundCtx<NoiseT>& c, int n) {
    const int e = c.vlist[n];
    const int pix = entry_pixel(e, c.invK), k = e - pix * c.K;
    const float x = c.xs[n];
    uint32_t w[4];
    float p, t;
    const int F = compound_flips(c, k, pix, x, w, p, t);
    float r = 0.0f;
    if (F > 0) {
        uint32_t q = c.c0;
        int idx = 1;
#pragma unroll 1
        for (int i = 0; i < F; ++i) {
            if (idx == 4) {
                ++q;
                c.noise.words(q, (uint32_t)k, c.pix0 + pix, w);
                idx = 0;
            }
            const uint32_t word = idx == 0 ? w[0] : idx == 1 ? w[1] : idx == 2 ? w[2] : w[3];
            ++idx;
            const float v = ((float)word + 1.0f) * 2.3283064365386963e-10f;  // (0, 1]
            // T = -Phi^-1(v p) >= t:  Phi(-T) = v p
            r += fmaxf(1.4142135623730951f * erfcinvf(2.0f * v * p), t);
        }
    }
    c.cnt[n] = (uint16_t)((x >= 0.0f) ? c.n_loc - F : F);
    c.rs[n] = r;
}

// forward-only render: the count of entry n alone.  F is drawn from the same counter word as in compound_entry, so the
// count is the training forward's; the tail normals, which only feed rs, are not drawn
template <class NoiseT>
static __device__ __noinline__ void compound_count_entry(const CompoundCtx<NoiseT>& c, int n) {
    const int e = c.vlist[n];
    const int pix = entry_pixel(e, c.invK), k = e - pix * c.K;
    const float x = c.xs[n];
    uint32_t w[4];
    float p, t;
    const int F = compound_flips(c, k, pix, x, w, p, t);
    c.cnt[n] = (uint16_t)((x >= 0.0f) ? c.n_loc - F : F);
}

// The listed entries (blist[0], blist[-1], ..., blist[-(nb-1)]: compact indices, stored downwards) in warp passes of
// entries with a similar expected number of flips, so that the lanes of a pass loop about equally long: three sweeps
// over the list (|x| < x_b2: many flips, < x_b3: some, rest: rarely any), each compacting its entries through a
// 64-slot ring in shared memory and running a pass whenever 32 are pending.
// ENTRY: compound_entry, or compound_count_entry for the forward-only render.
template <class NoiseT, void (*ENTRY)(const CompoundCtx<NoiseT>&, int)>
__device__ __forceinline__ void compound_sweep(const CompoundCtx<NoiseT>& c, const uint16_t* blist, int nb, float x_b2,
                                               float x_b3, uint16_t* ring) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    if (nb <= 32) {
        if (lane < nb) ENTRY(c, blist[-lane]);
        return;
    }
#pragma unroll 1
    for (int b = 0; b < 3; ++b) {
        int have = 0, done = 0;
#pragma unroll 1
        for (int base = 0; base < nb; base += 32) {
            const int li = base + lane;
            const int n = li < nb ? blist[-li] : 0;
            const float ax = fabsf(c.xs[n]);
            const bool sel = li < nb && (ax < x_b2 ? 0 : ax < x_b3 ? 1 : 2) == b;
            const unsigned m = __ballot_sync(FULL, sel);
            if (sel) ring[(have + __popc(m & lt)) & 63] = (uint16_t)n;
            have += __popc(m);
            __syncwarp();
            if (have - done >= 32) {
                ENTRY(c, ring[(done + lane) & 63]);
                done += 32;
                __syncwarp();
            }
        }
        if (lane < have - done) ENTRY(c, ring[(done + lane) & 63]);
        __syncwarp();
    }
}

template <class NoiseT>
static __device__ __noinline__ void rast_compound_list(const CompoundCtx<NoiseT>& c, const uint16_t* blist, int nb, float x_b2,
                                                       float x_b3, uint16_t* ring) {
    compound_sweep<NoiseT, compound_entry<NoiseT>>(c, blist, nb, x_b2, x_b3, ring);
}

template <class NoiseT>
static __device__ __noinline__ void rast_compound_count_list(const CompoundCtx<NoiseT>& c, const uint16_t* blist, int nb,
                                                             float x_b2, float x_b3, uint16_t* ring) {
    compound_sweep<NoiseT, compound_count_entry<NoiseT>>(c, blist, nb, x_b2, x_b3, ring);
}

// ------------------------------------------------------------------------------------------------
// per-pixel preparation, G lanes per pixel, all pixels of the tile at once.
// In:  zs[n] = raw zbuf, cnt[n] = hit count over ALL coverage samples.   Out: zs[n] = zeta_k.
// Values returned are uniform over the lanes of a pixel's group.
// ------------------------------------------------------------------------------------------------
struct PixPrep {
    float zmax;      // max(max_k zi_k, eps)
    float zimax;     // max_k zi_k (padded entries contribute zi = 0)
    float prod_nz;   // prod over entries with P != 1 of (1 - P)
    float zeta_max;  // max_j zeta_j (incl. background)
    float zbg;       // zeta_K = eps - zmax
    int argzi;       // argmax_k zi_k (first index)
    int nzero;       // number of entries with P == 1
    int a0;          // argmax_j zeta_j (first index), K = background
    int kpad;        // first padded k, K if none
};

__device__ __forceinline__ PixPrep prep_pixels(int p, int lig, int G, bool pvalid, int K, const int* vstart,
                                               const uint16_t* vlist, const uint16_t* cnt, float* zs, float zn,
                                               float zf, int S_rast, float gal, float eps) {
    const int vs = pvalid ? vstart[p] : 0, ve = pvalid ? vstart[p + 1] : 0;
    const int nv = ve - vs;
    const int e_base = p * K;
    float zimax = -CUDART_INF_F;
    int argzi = 0x7fffffff;
    float prod = 1.0f;
    int nzero = 0;
    int kpad = 0x7fffffff;
    const float denom = zf - zn;
    const float fS = (float)S_rast;
#pragma unroll 1
    for (int n = vs + lig; n < ve; n += G) {
        const int k = (int)vlist[n] - e_base;
        const float pk = (float)cnt[n] / fS;
        const float om = 1.0f - pk;
        if (om == 0.0f) nzero++; else prod *= om;
        const float zi = __fdiv_rn(zf - zs[n], denom);
        zs[n] = zi;
        if (zi > zimax) {
            zimax = zi;
            argzi = k;
        }
        if (k != n - vs) kpad = min(kpad, n - vs);
    }
    __syncwarp();
    group_argmax(zimax, argzi, G);
    prod = group_prod(prod, G);
    nzero = group_sum_i(nzero, G);
    kpad = group_min_i(kpad, G);
    if (kpad == 0x7fffffff) kpad = nv;  // valid entries are a prefix: first padded index is nv (== K: none)
    if (kpad < K) {
        // masked entries have zi = (..)*0 = 0 and take part in the max (smoothagg.py:198-199)
        if (0.0f > zimax || (0.0f == zimax && kpad < argzi)) {
            zimax = 0.0f;
            argzi = kpad;
        }
    }
    const float zmax = fmaxf(zimax, eps);
    const float zbg = __fadd_rn(eps, -zmax);
    float best = -CUDART_INF_F;
    int a0 = 0x7fffffff;
#pragma unroll 1
    for (int n = vs + lig; n < ve; n += G) {
        const int k = (int)vlist[n] - e_base;
        const int c = cnt[n];
        float z = -CUDART_INF_F;
        if (c != 0) {
            const float lg = (c == S_rast) ? 0.0f : logf_exact((float)c / fS);
            z = __fadd_rn(__fadd_rn(__fmul_rn(gal, lg), zs[n]), -zmax);
        }
        zs[n] = z;
        if (z > best) {
            best = z;
            a0 = k;
        }
    }
    __syncwarp();
    group_argmax(best, a0, G);
    if (!(best >= zbg)) {  // background wins ties only against nothing: it is the LAST index
        best = zbg;
        a0 = K;
    }
    PixPrep pi;
    pi.zmax = zmax;
    pi.zimax = zimax;
    pi.prod_nz = prod;
    pi.nzero = nzero;
    pi.argzi = argzi;
    pi.a0 = a0;
    pi.zeta_max = best;
    pi.zbg = zbg;
    pi.kpad = kpad;
    return pi;
}

// logits further than this below the largest one can never win a sample (bounded noise); the absolute
// term covers the rounding of z + gamma*n
__device__ __forceinline__ float live_cut(float gamma, float zeta_max, bool bounded) {
    return bounded ? 2.0f * gamma * kNoiseAbsMax * 1.0001f + 4e-7f * fmaxf(1.0f, fabsf(zeta_max)) : CUDART_INF_F;
}

}  // namespace pert
