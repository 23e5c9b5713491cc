// Counter-based noise for the perturbed shader: Philox4x32-10 (Salmon et al., SC'11) + Box-Muller.
//
// One Philox call yields the four standard normals of samples 4q..4q+3 for ONE noise coordinate:
//     counter = (q, slot, pixel_lo, pixel_hi | stage << 31),  key = seed
// where `pixel` is the GLOBAL pixel index (batch shards of one job draw the same noise as the
// unsharded job), `slot` is the face index k (coverage stage) or logit index j (aggregation stage,
// j = K is the background), and `q = s >> 2`.  Nothing sample-sized is ever stored: forward and
// backward regenerate the same values from the same counters.
//
// Replaces the two materialised draws of the reference, torch.normal(zeros(S,N,H,W,K)) at
// randomras/smoothrast.py:21 and torch.normal(zeros(S,N,H,W,K+1)) at randomras/smoothagg.py:21.
#pragma once
#include <cstdint>

namespace pert {

// Every uniform is built from the top 23 bits of a Philox word (mantissa trick, no I2F on the
// quarter-rate conversion pipe): u in [2^-23, 1], so |n| <= sqrt(-2 ln 2^-23) = 5.647 for every value
// box_muller() can return; the kernels use this bound to skip draws that cannot change any output
// bit.  (The truncated tail has probability 1.6e-8 per draw.)
constexpr float kNoiseAbsMax = 5.66f;

template <int ROUNDS>
__device__ __forceinline__ void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                           uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1;
        c3 = (uint32_t)p0;
        c0 = n0;
        c2 = n2;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0;
    out[1] = c1;
    out[2] = c2;
    out[3] = c3;
}

// top 23 bits of a word as a float in [1, 2)
__device__ __forceinline__ float mant12(uint32_t x) { return __uint_as_float((x >> 9) | 0x3f800000u); }

__device__ __forceinline__ float mufu_lg2(float x) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float mufu_sqrt(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float mufu_sin(float x) {
    float r;
    asm("sin.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float mufu_cos(float x) {
    float r;
    asm("cos.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// Two standard normals from two 32-bit words: u = 2 - mant12(a) in [2^-23, 1], radius =
// sqrt(-2 ln u) (MUFU.LG2 + MUFU.SQRT), angle = 2 pi (mant12(b) - 1.5) in [-pi, pi) (MUFU.SIN /
// MUFU.COS).  u is never denormal, so the .ftz forms are exact substitutes.
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& n0, float& n1) {
    const float u = 2.0f - mant12(a);
    const float rad = mufu_sqrt(-1.3862943611198906f * mufu_lg2(u));
    const float ang = fmaf(mant12(b), 6.283185307179586f, -9.42477796076938f);
    n0 = rad * mufu_cos(ang);
    n1 = rad * mufu_sin(ang);
}

// ROUNDS = 10 is the generator of the Random123 paper and cuRAND; 7 rounds is the paper's Crush-resistant minimum
// (PERT_F_PHILOX7: 30 % fewer multiply / xor pairs per call, another stream).
template <int ROUNDS>
struct PhiloxNoiseT {
    uint32_t k0, k1;
    uint32_t stage_bit;  // 0 or 0x80000000
    int64_t pixel_offset;

    __host__ __device__ __forceinline__ PhiloxNoiseT(uint64_t seed, int stage, int64_t pixel_off)
        : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), stage_bit(stage ? 0x80000000u : 0u), pixel_offset(pixel_off) {}

    // normals of samples 4q..4q+3 for (pixel_local, slot)
    __device__ __forceinline__ void get4(uint32_t q, uint32_t slot, int64_t pixel_local, float (&n)[4]) const {
        const uint64_t gp = (uint64_t)(pixel_local + pixel_offset);
        uint32_t r[4];
        philox4x32<ROUNDS>(q, slot, (uint32_t)gp, ((uint32_t)(gp >> 32) & 0x7fffffffu) | stage_bit, k0, k1, r);
        box_muller(r[0], r[1], n[0], n[1]);
        box_muller(r[2], r[3], n[2], n[3]);
    }
    // the raw Philox words of (q, slot, pixel): r[0],r[1] make samples 4q, 4q+1 and r[2],r[3] make 4q+2, 4q+3
    __device__ __forceinline__ void words(uint32_t q, uint32_t slot, int64_t pixel_local, uint32_t (&r)[4]) const {
        const uint64_t gp = (uint64_t)(pixel_local + pixel_offset);
        philox4x32<ROUNDS>(q, slot, (uint32_t)gp, ((uint32_t)(gp >> 32) & 0x7fffffffu) | stage_bit, k0, k1, r);
    }
    // device-side seed (pert_problem.seed_device): the effective seed is seed ^ v
    __device__ __forceinline__ void mix(uint64_t v) {
        k0 ^= (uint32_t)v;
        k1 ^= (uint32_t)(v >> 32);
    }
    static constexpr bool kBounded = true;
};
using PhiloxNoise = PhiloxNoiseT<10>;
using PhiloxNoise7 = PhiloxNoiseT<7>;

// Standard Cauchy noise from the same counters: tan(pi (u - 1/2)), clamped to +-1e7 like the reference
// (randomras/smoothrast.py:22-24, smoothagg.py:25-27).  Heavy tails: nothing can be skipped (not bounded).
struct PhiloxCauchy {
    PhiloxNoise base;
    __host__ __device__ __forceinline__ PhiloxCauchy(uint64_t seed, int stage, int64_t pixel_off) : base(seed, stage, pixel_off) {}
    __device__ __forceinline__ void get4(uint32_t q, uint32_t slot, int64_t pixel_local, float (&n)[4]) const {
        uint32_t r[4];
        base.words(q, slot, pixel_local, r);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const float a = (mant12(r[t]) - 1.5f) * 3.14159265358979f;  // [-pi/2, pi/2)
            n[t] = fminf(fmaxf(__fdividef(mufu_sin(a), mufu_cos(a)), -1e7f), 1e7f);
        }
    }
    __device__ __forceinline__ void mix(uint64_t v) { base.mix(v); }
    static constexpr bool kBounded = false;
};

// Uniform noise on [-1/2, 1/2) (the reference's UniformAgg: torch.distributions.Uniform(-0.5, 0.5), smoothagg.py:28-30)
// and standard Gumbel noise -log(-log u) (smoothagg.py:22-24) from the same counters.  Forward only: the reference has
// no backward for either (smoothagg.py:64-67 prints "noise_type not implemented").  Not treated as bounded by the
// kernels' skipping rules (those are written for the Gaussian bound).
struct PhiloxUniform {
    PhiloxNoise base;
    __host__ __device__ __forceinline__ PhiloxUniform(uint64_t seed, int stage, int64_t pixel_off) : base(seed, stage, pixel_off) {}
    __device__ __forceinline__ void get4(uint32_t q, uint32_t slot, int64_t pixel_local, float (&n)[4]) const {
        uint32_t r[4];
        base.words(q, slot, pixel_local, r);
#pragma unroll
        for (int t = 0; t < 4; ++t) n[t] = mant12(r[t]) - 1.5f;
    }
    static constexpr bool kBounded = false;
};
struct PhiloxGumbel {
    PhiloxNoise base;
    __host__ __device__ __forceinline__ PhiloxGumbel(uint64_t seed, int stage, int64_t pixel_off) : base(seed, stage, pixel_off) {}
    __device__ __forceinline__ void get4(uint32_t q, uint32_t slot, int64_t pixel_local, float (&n)[4]) const {
        uint32_t r[4];
        base.words(q, slot, pixel_local, r);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const float u = 2.0f - mant12(r[t]);  // (0, 1]
            n[t] = -logf(fmaxf(-logf(u), 1e-30f));
        }
    }
    static constexpr bool kBounded = false;
};

// score of the noise density used by the gradient estimators: -d/dn log p(n)
//   Gaussian: n   (smoothrast.py:46, smoothagg.py:51-53)     Cauchy: 2n / (1 + n^2)   (smoothrast.py:49, smoothagg.py:58-59)
// SCORE = 0 / 1 is a compile-time parameter of the kernels, separate from the noise source: explicit noise works with
// either law
template <int SCORE>
__device__ __forceinline__ float noise_score(float n) {
    return SCORE == 0 ? n : __fdividef(2.0f * n, 1.0f + n * n);
}

// Explicit noise tensor (S, P, slots), e.g. the reference's own draws: used for exact-noise parity.
struct ExplicitNoise {
    const float* base;
    int64_t P;
    int32_t slots;
    int32_t S;
    __device__ __forceinline__ void mix(uint64_t) {}

    __device__ __forceinline__ void get4(uint32_t q, uint32_t slot, int64_t pixel_local, float (&n)[4]) const {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int64_t s = (int64_t)q * 4 + t;
            n[t] = (s < S) ? __ldg(base + (s * P + pixel_local) * slots + slot) : 0.0f;
        }
    }
    static constexpr bool kBounded = false;
};

// Radius bound on the raw word: box_muller(a, .) returns |n| < t for every angle whenever
// (a >> 9) < radius_gate(t).  u = 1 - (a >> 9) 2^-23 exactly, and rad < t  <=>  u > exp(-t^2/2); the
// 1.001 factor on exp(.) and the -2 cover the MUFU approximation errors of rad, cos and sin by a wide
// margin (a conservative gate only costs a wasted Box-Muller, never a wrong sample).
__device__ __forceinline__ uint32_t radius_gate(float t) {
    const float e = exp2f(-0.72134752f * t * t) * 1.001f;
    const float g = (1.0f - e) * 8388608.0f - 2.0f;
    return g > 0.0f ? (uint32_t)g : 0u;
}

}  // namespace pert
