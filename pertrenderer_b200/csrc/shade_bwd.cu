// Fused backward of the perturbed shader (pert_shade_bwd in include/pertshade.h).
//
// Reference path (autograd of smooth_rgb_blend, randomras/random_rasterizer.py:34-56):
//   randomArgmax.backward     randomras/smoothagg.py:45-73
//   cat / max / clamp, log_corrected / prod_corrected backward   randomras/smoothagg.py:198-202, 303-337
//   prod backward (alpha), mask backward                          randomras/random_rasterizer.py:47-48
//   randomHeaviside.backward  randomras/smoothrast.py:40-59
//
// One warp per tile of tp pixels.  Phases of a tile:
//   0  zero-fill the tile's rows of grad_dists / grad_zbuf / grad_colors (128-bit stores), scan
//      pix_to_face -> compact list of valid entries; zbuf and saved state only for those
//   1  per-pixel logits (same arithmetic as forward)
//   2  pixels where some sample left the unperturbed winner: histogram of the saved winners, g_j,
//      c_s = g[a_s] - g[a_0]
//   3  score sums acc_j = sum_s c_s V_sj, t2_j = sum_s c_s V_sj^2 over (pixel, logit) pairs, noise
//      regenerated from the Philox counters
//   4  chain rule per valid entry -> scattered stores over the zero-filled rows; scalar partials
#include <climits>
#include "kernels.h"
#include "tile.cuh"

namespace pert {

// Active pixels whose per-sample c_s are staged at a time (<= 8: the pair codes hold the rank in 3 bits; shared memory =
// occupancy).  In the fallback pass that is the pixels of its tiles: one batch (4 rows of c_s would buy a thirteenth CTA per
// SM and lose more to the second batch: profiles/r2_notes.md)
constexpr int kNab = 8;

// lean (the passes' time follows the warps an SM holds, i.e. the bytes of this layout): the pair list takes over the counts
// array (phase 4 reads the counts from global memory instead)
void bwd_smem_layout(int tp, int K, int cap, int sc, int nchunks, int win_bytes, bool compact, bool lean, SmemLayout& L) {
    const size_t ns = compact ? (size_t)cap + 2 * tp : (size_t)tp * (K + 1);
    Carver cv(L);
    cv.take(cap, 2);  // vlist
    cv.take(ns > (size_t)cap ? ns : (size_t)cap, 4);  // zs, then accs (the logits are dead once the live ones are marked)
    cv.take(lean && ns > (size_t)cap ? ns : (size_t)cap, 2);  // cnt (lean: then the pair list)
    cv.take(ns, 4);   // hj
    cv.take(ns, 4);   // gsel (| t2s when there is one sample chunk)
    cv.take(nchunks > 1 ? ns : 0, 4);  // t2s
    cv.take(lean ? 0 : ns, 2);   // pairs
    cv.take((size_t)(tp < kNab ? tp : kNab) * sc, 4);  // cs
    cv.take(tp + 1, 4);           // vstart
    cv.take(tp, 4);               // pa0
    cv.take(tp, 4);               // pg0
    cv.take(compact ? tp : 0, 4);  // psb (dense per-logit arrays: the slot base is p * (K + 1))
    cv.take(compact ? tp : 0, 4);  // pnv
    cv.take(tp, 1);               // apx
    cv.take(nchunks == 1 ? (size_t)tp * sc * win_bytes : 0, 1);  // wst
}

// GT = lanes per pixel as a compile-time constant (1, 2, 4, 8), or 0 to read it from the launch record.
// PHASED = false is the production instantiation: both phases in one launch, histogram rebuilt from the
// saved winners (the phase-split code of the sample-sharded job is compiled out to keep the hot code small).
// FACE = true: colours gathered through pix_to_face from pb.face_colors, grad scattered by atomics
// COMPACT = true (sparse-first mode): the per-logit arrays are indexed by the position of the logit
// among the pixel's valid entries (plus a background and a masked-logits slot) instead of densely by j,
// and every array holds a.L.cap valid entries; tiles with more go to the fallback pass.
// BLOB = true (only with COMPACT): the compact valid list and the per-pixel logit summary come from the tile
// blob forward saved (common.cuh) instead of a re-scan of pix_to_face and a recomputation of the logits.
// SCORE = the score psi of the aggregation noise (philox.cuh noise_score): acc_j = sum_s c_s psi(V_sj) and
// t2_j = sum_s c_s V_sj psi(V_sj); 0 Gaussian (psi(n) = n), 1 Cauchy.
// WOVR = true (PERT_F_NO_VR, randomArgmax_wovr smoothagg.py:75-141): c_s = g[a_s] without the control variate g[a_0].
// Samples that picked a0 contribute, so every valid pixel is worked on, including those whose samples all picked a0
// (forward wrote no winners row for them when a0 was their only live logit: a_s = a0 is known) and the pixels
// without any valid entry (the background wins every sample; their only output is the gamma term, whose norm runs
// over all K + 1 logits).  Every V_sj of every logit is regenerated (per-sample noise, dense per-logit arrays).
template <class NoiseA, int GT, bool PHASED, bool FACE, bool COMPACT, bool BLOB, int SCORE = 0, bool WOVR = false>
__device__ __forceinline__ void shade_bwd_tile(const BwdArgs& a, const NoiseA& noise_a, const int64_t tile,
                                               const int64_t prow /* row of the scalar partials */,
                                               unsigned char* smem_raw, const int lane) {
    const pert_problem& pb = a.pb;
    const int G = GT ? GT : a.L.G;
    const int gshift = GT ? (GT == 16 ? 4 : GT == 8 ? 3 : GT == 4 ? 2 : GT == 2 ? 1 : 0) : a.L.gshift;
    const int K = pb.K, K1 = K + 1, tp = 32 >> gshift, sc = a.L.sc;
    const uint32_t flags = pb.flags;
    const bool do_sample = !PHASED || (flags & PERT_PH_BWD_SAMPLE), do_finish = !PHASED || (flags & PERT_PH_BWD_FINISH);
    const int32_t* const ghist = PHASED ? a.hist : nullptr;
    const bool no_skip = flags & PERT_F_NO_SKIP;
    // how the noise of logits that can never win (zero-mean, independent of everything) is handled; the one-draw
    // shortcut rests on sum_s c_s V_sj being normal, which holds for the Gaussian score only
    const bool per_sample = WOVR || SCORE != 0 || !NoiseA::kBounded || no_skip || (flags & PERT_F_PER_SAMPLE_NOISE);
    const bool drop_dead = !per_sample && (flags & PERT_F_SKIP_DEAD_NOISE);
    float p_sigma = 0.f, p_gamma = 0.f, p_q = 0.f;

    const int64_t pix0 = tile * tp;
    const int npx = (int)min((int64_t)tp, a.L.P - pix0);
    const int E = npx * K;
    const int64_t g0 = pix0 * K;
    const int p = lane >> gshift, lig = lane & (G - 1);
    const bool pvalid = p < npx;
    const int64_t gp = pix0 + p;
    const unsigned lt = (1u << lane) - 1u;
    const int sa_loc = a.L.sa_loc;
    const int wb = a.L.win_bytes;

    Taker cv(smem_raw, a.L.sm);  // layout: bwd_smem_layout
    const int cap = a.L.cap;
    uint16_t* vlist = cv.take<uint16_t>();
    float* zs = cv.take<float>();
    uint16_t* cnt = cv.take<uint16_t>();
    // per-logit arrays.  Slot of logit j of pixel p: dense p*K1 + j, or (COMPACT) vstart[p] + 2p + idx with
    // idx = position among the pixel's valid entries, nvp = background, nvp + 1 = all masked logits together
    // winner histogram (active pixels); INT_MIN marks the logits that can never win a sample (their zeta is not
    // needed again after phase 2, which lets the score sums take over the zeta array: shared memory = occupancy)
    int* hj = cv.take<int>();
    float* gsel = cv.take<float>();  // g_j = <G_rgb, colour_j> of the logits that can win
    float* accs = zs;                // sum_s c_s V_sj (from the end of phase 2 on)
    // sum_s c_s V_sj^2: g_j is dead once the c_s of the (only) chunk are staged, so it reuses that array
    float* t2s_own = cv.take<float>();
    float* t2s = a.L.nchunks > 1 ? t2s_own : gsel;
    // (pixel, logit) pairs that need per-sample noise: logit j (or, COMPACT, its position among the pixel's valid
    // entries) in bits 0-9 (K <= 1023), the pixel's rank among the staged active pixels in bits 10-12 (kNab <= 8)
    uint16_t* pairs_own = cv.take<uint16_t>();
    const bool lean = a.L.lean;
    uint16_t* pairs = lean ? cnt : pairs_own;
    float* cs = cv.take<float>();  // c_s of the current sample chunk, per active pixel
    int* vstart = cv.take<int>();
    int* pa0 = cv.take<int>();
    float* pg0 = cv.take<float>();
    int* psb = cv.take<int>();  // slot base of every pixel
    int* pnv = cv.take<int>();  // number of valid entries | 0x10000 if they are NOT a prefix 0..nvp-1 of K
    uint8_t* apx = cv.take<uint8_t>();
    // single-chunk jobs: the tile's saved winners (tp rows of sa_loc entries, contiguous) are copied to
    // shared memory asynchronously at the very start, off the critical path
    const bool early_w = a.L.nchunks == 1 && ((sa_loc * wb) & 15) == 0 && do_sample && (((uintptr_t)a.winners) & 15) == 0;
    unsigned char* wst = cv.take<unsigned char>();
    if (early_w) {
        const unsigned char* src = reinterpret_cast<const unsigned char*>(a.winners) + pix0 * sa_loc * wb;
        const int nbytes = npx * sa_loc * wb;
#pragma unroll 1
        for (int o = lane * 16; o < nbytes; o += 32 * 16) cp_async16(wst + o, src + o);
    }

    // ---- phase 0 -----------------------------------------------------------------------------------
    // per-pixel inputs do not depend on the scan: issue their loads first
    float4 Gi = make_float4(0.f, 0.f, 0.f, 0.f);
    float zn = 1.0f, zf = 100.0f;
    int pstate = K;
    if (pvalid) {
        Gi = __ldg(reinterpret_cast<const float4*>(a.grad_image) + gp);
        const int b = pb.depth_len > 1 ? batch_of(pix0, p, a.L.HW) : 0;
        zn = __ldg(pb.znear + b);
        zf = __ldg(pb.zfar + b);
        pstate = a.pixstate[gp];
    }
    const int32_t* const bl = BLOB ? a.blob + tile * (int64_t)blob_words(tp, cap) : nullptr;
    const int nv = BLOB ? __ldg(bl) : scan_valid(pb.pix_to_face + g0, E, a.L.vec_ok, vlist, cap);
    const bool overflow = COMPACT && (BLOB ? nv < 0 : nv > cap);
    if (!overflow) {
        // this pass owns the tile: its output rows start as zeros, valid entries are scattered over them later
        if (do_finish) {
            zero_fill(a.grad_dists + g0, E, a.L.vec_ok);
            zero_fill(a.grad_zbuf + g0, E, a.L.vec_ok);
            if (a.grad_colors && !FACE) zero_fill(a.grad_colors + g0 * 3, E * 3, a.L.vec_ok);
        } else {
            zero_fill(a.acc + pix0 * K1, npx * K1, false);
            if (lane < npx) {
                a.pixstat[(pix0 + lane) * 2] = 0.f;
                a.pixstat[(pix0 + lane) * 2 + 1] = 0.f;
            }
        }
    }
    if (overflow) {
        // more valid entries than the compact arrays hold: the fallback pass redoes this tile
        if (lane == 0) a.worklist[4 + atomicAdd(a.worklist, 1)] = (int32_t)tile;
    } else if (nv > 0 || WOVR) {
        const float gal = a.L.gal;
        PixPrep pi;
        if constexpr (BLOB) {
            // ---- phase 1 (from forward's blob) -------------------------------------------------------
            const float* const colors_t = pb.colors + g0 * 3;
            const float* const rsum_t = a.rsum + g0;
            for (int i = lane; i <= tp; i += 32) vstart[i] = __ldg(bl + 1 + i);
            uint32_t* const vl32 = reinterpret_cast<uint32_t*>(vlist);
            uint32_t* const cn32 = reinterpret_cast<uint32_t*>(cnt);
            const int nw = (nv + 1) >> 1;
#pragma unroll 1
            for (int i = lane; i < nw; i += 32) {
                const uint32_t v2 = (uint32_t)__ldg(bl + blob_vlist_off(tp) + i);
                vl32[i] = v2;
                cn32[i] = (uint32_t)__ldg(bl + blob_cnt_off(tp, cap) + i);
                // needed a few round trips later (g_j of the logits that can win; chain rule): start them now
                const int e0 = v2 & 0xffff, e1 = v2 >> 16;
                if (!FACE) prefetch_l1(colors_t + e0 * 3);
                prefetch_l1(rsum_t + e0);
                if (2 * i + 1 < nv) {
                    if (!FACE) prefetch_l1(colors_t + e1 * 3);
                    prefetch_l1(rsum_t + e1);
                }
            }
#pragma unroll 1
            for (int i = lane; i < nv; i += 32) zs[i] = __int_as_float(__ldg(bl + blob_zeta_off(tp, cap) + i));
            if (pvalid) {
                const int32_t* const bp = bl + blob_pix_off(tp) + 6 * p;
                pi.zmax = __int_as_float(__ldg(bp));
                pi.zimax = __int_as_float(__ldg(bp + 1));
                pi.prod_nz = __int_as_float(__ldg(bp + 2));
                pi.zeta_max = __int_as_float(__ldg(bp + 3));
                const int w4 = __ldg(bp + 4), w5 = __ldg(bp + 5);
                pi.argzi = w4 & 0xffff;
                pi.a0 = w4 >> 16;
                pi.nzero = w5 & 0xffff;
                pi.kpad = w5 >> 16;
            } else {
                pi.zmax = pb.eps;
                pi.zimax = 0.f;
                pi.prod_nz = 1.f;
                pi.zeta_max = 0.f;
                pi.argzi = pi.a0 = pi.nzero = pi.kpad = 0;
            }
            pi.zbg = __fadd_rn(pb.eps, -pi.zmax);
            __syncwarp();
        } else {
            __syncwarp();
            pixel_ranges(vlist, nv, K, tp, vstart);
            {
                const float* const zbuf_t = pb.zbuf + g0;
                const uint16_t* const counts_t = a.counts + g0;
                const float* const colors_t = pb.colors + g0 * 3;
                const float* const rsum_t = a.rsum + g0;
#pragma unroll 1
                for (int n = lane; n < nv; n += 32) {
                    const int e = vlist[n];
                    zs[n] = __ldg(zbuf_t + e);
                    cnt[n] = counts_t[e];
                    // needed a few round trips later (g_j of the logits that can win; chain rule): start them now
                    if (!FACE) prefetch_l1(colors_t + e * 3);
                    prefetch_l1(rsum_t + e);
                }
            }
            __syncwarp();

            // ---- phase 1 ---------------------------------------------------------------------------
            pi = prep_pixels(p, lig, G, pvalid, K, vstart, vlist, cnt, zs, zn, zf, pb.S_rast, gal, pb.eps);
        }
        const int vs = pvalid ? vstart[p] : 0, ve = pvalid ? vstart[p + 1] : 0;
        const int nvp = ve - vs;
        const int a0 = pi.a0;
        // a pixel whose samples all picked a0 has c_s = 0 for every s: every score sum is exactly 0
        // (and forward wrote no winners row for it); without the control variate c_s = g[a0] there
        const bool act = pvalid && do_sample && (WOVR || (pstate & 0x8000));
        const int sb = COMPACT ? vs + 2 * p : p * K1;                  // this pixel's slots
        const int slot_pad = COMPACT ? sb + nvp + 1 : sb + pi.kpad;     // where the masked logits' joint draw goes
        const bool prefix = pi.kpad == nvp;                             // valid entries are k = 0..nvp-1
        // slot of logit j of pixel pp (j = a saved winner or a0: a valid entry or the background)
        auto slot_of = [&](int pp, int j) -> int {
            if (!COMPACT) return pp * K1 + j;
            const int base = psb[pp], info = pnv[pp], n = info & 0xffff;
            if (j == K) return base + n;
            if (!(info & 0x10000)) return base + j;
            const int lo = vstart[pp];  // holes in the mask: find the entry
            return base + lower_bound_u16(vlist, lo, lo + n, pp * K + j) - lo;
        };
        const float floor_v = pi.zeta_max - live_cut(pb.gamma, pi.zeta_max, NoiseA::kBounded && !no_skip);
        float t2sum = 0.f, csum = 0.f;
        const float* gacc = a.acc + gp * K1;  // FINISH-only: sums over all sample shards
        const float* const colors_p = pb.colors + gp * K * 3;
        const float* const fcol = FACE ? pb.face_colors : nullptr;  // per-face colours gathered through pix_to_face
        const int64_t* const p2f_p = pb.pix_to_face + gp * K;
        __syncwarp();

        // ---- phase 2 -------------------------------------------------------------------------------
        const unsigned actb = __ballot_sync(FULL, act && lig == 0);
        const int na = __popc(actb);
        const int my_ai = __popc(actb & ((1u << (p * G)) - 1u));
        if (na > 0) {
            // g_j of every logit that can win (the saved winners are among them) and cleared sums
            if (act && lig == 0) {
                apx[my_ai] = (uint8_t)p;
                // WOVR: bit 16 = every sample picked a0, the saved winners row is not read
                pa0[p] = (WOVR && !(pstate & 0x8000)) ? a0 | 0x10000 : a0;
                if (COMPACT) {
                    psb[p] = sb;
                    pnv[p] = nvp | (prefix ? 0 : 0x10000);
                }
            }
            const int nsl = COMPACT ? nvp + 2 : K1;
            if (act) {
#pragma unroll 1
                for (int j = lig; j < nsl; j += G) hj[sb + j] = 0;
            }
            __syncwarp();
            if (act) {
#pragma unroll 1
                for (int idx = lig; idx <= nvp; idx += G) {
                    const int j = idx < nvp ? (int)vlist[vs + idx] - p * K : K;
                    const float z = idx < nvp ? zs[vs + idx] : pi.zbg;
                    const int sl = COMPACT ? sb + idx : sb + j;
                    if (z > -CUDART_INF_F && z >= floor_v) {
                        float gj;
                        if (j < K) {
                            const float* c = fcol ? fcol + 3 * (int)__ldg(p2f_p + j) : colors_p + j * 3;
                            gj = Gi.x * __ldg(c) + Gi.y * __ldg(c + 1) + Gi.z * __ldg(c + 2);
                        } else {
                            gj = Gi.x * pb.background[0] + Gi.y * pb.background[1] + Gi.z * pb.background[2];
                        }
                        gsel[sl] = gj;
                        if (j == a0) pg0[p] = gj;
                    } else {
                        hj[sl] = INT_MIN;  // can never win
                    }
                }
            }
            __syncwarp();  // every lane has read its logits: the array becomes the score sums
            if (act) {
#pragma unroll 1
                for (int j = lig; j < nsl; j += G) accs[sb + j] = 0.f;
            }
            __syncwarp();

            // ---- phase 3: one pass over the saved winners per sample chunk: histogram + c_s, then the
            //      score sums of the pairs ------------------------------------------------------------------
            const int qb = pb.s_agg_begin >> 2;
            if (early_w) {
                cp_async_wait_all();
                __syncwarp();
            }
            float C2 = 0.f;
            // active pixels are processed kNab at a time: the c_s staging buffer holds kNab rows
#pragma unroll 1
            for (int b0 = 0; b0 < na; b0 += kNab) {
            const int nb = min(kNab, na - b0);
            const bool mine = act && my_ai >= b0 && my_ai < b0 + kNab;
            // the (pixel, logit) pairs of this batch that need per-sample noise
            int np2 = 0;
            {
                const int span = (!COMPACT && per_sample) ? K1 : nvp + 1;
                const int iters = warp_max_i(mine ? (span + G - 1) / G : 0);
#pragma unroll 1
                for (int it = 0; it < iters; ++it) {
                    const int idx = it * G + lig;
                    bool want = false;
                    int j = idx;
                    if (mine && idx < span) {
                        if (!COMPACT && per_sample) {
                            want = true;  // every logit, dense in j
                        } else {
                            j = idx < nvp ? (int)vlist[vs + idx] - p * K : K;
                            want = hj[COMPACT ? sb + idx : sb + j] >= 0;  // can win (phase 2)
                        }
                    }
                    const unsigned wbal = __ballot_sync(FULL, want);
                    if (want) {
                        const int pos = np2 + __popc(wbal & lt);
                        pairs[pos] = (uint16_t)((COMPACT ? idx : j) | ((my_ai - b0) << 10));
                    }
                    np2 += __popc(wbal);
                }
            }
            __syncwarp();
            // lanes per pair: fewest issued instructions (see best_lane_shift), at most a.L.lpp
            const int lpp_shift = np2 == 0 ? 0 : best_lane_shift(np2, (min(sc, sa_loc) + 3) >> 2, a.L.lpp_shift);
            const int LPP = 1 << lpp_shift;
            const int lq = lane & (LPP - 1);
#pragma unroll 1
            for (int c0 = 0; c0 < sa_loc; c0 += sc) {  // c0 multiple of 32
                const int cn = min(sc, sa_loc - c0);
                const int cn4 = (cn + 3) & ~3;
#pragma unroll 1
                for (int ai = 0; ai < nb; ++ai) {
                    const int pp = apx[b0 + ai];
                    const float g0v = pg0[pp];
                    const int ppa0 = pa0[pp];
                    const int64_t wbase = (pix0 + pp) * sa_loc + c0;
#pragma unroll 1
                    for (int s = lane; s < cn4; s += 32) {
                        float c = 0.f;
                        if (s < cn) {
                            if constexpr (WOVR) {
                                const int pa = ppa0 & 0xffff;
                                const int w = (ppa0 & 0x10000) ? pa
                                              : early_w ? load_winner(wst, wb, pp * sa_loc + s) : load_winner(a.winners, wb, wbase + s);
                                if (w != pa) {
                                    const int ws = slot_of(pp, w);
                                    atomicAdd(&hj[ws], 1);
                                    c = gsel[ws];
                                } else {
                                    c = g0v;
                                }
                            } else {
                                const int w = early_w ? load_winner(wst, wb, pp * sa_loc + s) : load_winner(a.winners, wb, wbase + s);
                                if (w != ppa0) {  // a0 (the most frequent by far) is counted as the remainder
                                    const int ws = slot_of(pp, w);
                                    atomicAdd(&hj[ws], 1);
                                    c = gsel[ws] - g0v;
                                }
                            }
                        }
                        cs[ai * sc + s] = c;
                    }
                }
                __syncwarp();
                if (c0 + sc >= sa_loc) {
                    // all winners seen: histogram remainder, sum_s c_s and sum_s c_s^2 from the histogram (read
                    // g_j now: the pair loop below may reuse its array).  Group reductions run on every lane:
                    // pixels of one warp differ in `act`.
                    int others = 0;
                    float c1 = 0.f, c2 = 0.f;
                    if (mine) {
                        const float g0v = pg0[p];
#pragma unroll 1
                        for (int idx = lig; idx <= nvp; idx += G) {
                            const int j = idx < nvp ? (int)vlist[vs + idx] - p * K : K;
                            const int sl = COMPACT ? sb + idx : sb + j;
                            const int h = hj[sl];
                            if (h > 0 && j != a0) {
                                others += h;
                                const float d = WOVR ? gsel[sl] : gsel[sl] - g0v;
                                c1 += (float)h * d;
                                c2 += (float)h * d * d;
                            }
                        }
                    }
                    others = group_sum_i(others, G);
                    c1 = group_sum(c1, G);
                    c2 = group_sum(c2, G);
                    if (mine) {
                        csum = WOVR ? c1 + (float)(sa_loc - others) * pg0[p] : c1;  // the samples won by a0
                        C2 = c2;
                        if (lig == 0) hj[slot_of(p, a0)] = sa_loc - others;
                    }
                    __syncwarp();
                }
                const int nqc = cn4 >> 2;
#pragma unroll 1
                for (int it0 = 0; it0 < (np2 << lpp_shift); it0 += 32) {
                    const int it = it0 + lane;
                    const int pr = it >> lpp_shift;
                    const bool on = pr < np2;
                    const int code = on ? pairs[pr] : 0;
                    const int ai = code >> 10, cx = code & 1023;
                    const int pp = apx[b0 + ai];
                    int j = cx, ps;
                    if (COMPACT) {
                        const int nvq = pnv[pp] & 0xffff;
                        ps = psb[pp] + cx;
                        j = cx < nvq ? (int)vlist[vstart[pp] + cx] - pp * K : K;
                    } else {
                        ps = pp * K1 + cx;
                    }
                    float acc = 0.f, t2 = 0.f;
                    if (on) {
                        const float4* c4p = reinterpret_cast<const float4*>(cs + ai * sc);
#pragma unroll 1
                        for (int ql = lq; ql < nqc; ql += LPP) {
                            const float4 c4 = c4p[ql];
                            if (!no_skip && c4.x == 0.f && c4.y == 0.f && c4.z == 0.f && c4.w == 0.f) continue;
                            float nz[4];
                            noise_a.get4(qb + (c0 >> 2) + ql, j, pix0 + pp, nz);
                            const float cv0 = c4.x * noise_score<SCORE>(nz[0]), cv1 = c4.y * noise_score<SCORE>(nz[1]),
                                        cv2 = c4.z * noise_score<SCORE>(nz[2]), cv3 = c4.w * noise_score<SCORE>(nz[3]);
                            acc += (cv0 + cv1) + (cv2 + cv3);
                            t2 += (cv0 * nz[0] + cv1 * nz[1]) + (cv2 * nz[2] + cv3 * nz[3]);
                        }
                    }
#pragma unroll 1
                    for (int o = LPP >> 1; o > 0; o >>= 1) {
                        acc += __shfl_xor_sync(FULL, acc, o);
                        t2 += __shfl_xor_sync(FULL, t2, o);
                    }
                    if (on && lq == 0) {
                        if (c0 == 0) {
                            accs[ps] = acc;
                            t2s[ps] = t2;
                        } else {
                            accs[ps] += acc;
                            t2s[ps] += t2;
                        }
                    }
                }
                __syncwarp();
            }
            }  // batches of active pixels

            // ---- logits that can never win: their noise is independent of every a_s, so given c the sum
            //      sum_s c_s V_sj is N(0, sum_s c_s^2) exactly: ONE draw per logit instead of S_agg -------------
            {
                float t = 0.f;
                if (!COMPACT && per_sample) {
                    if (act) {
#pragma unroll 1
                        for (int j = lig; j < K1; j += G) t += t2s[p * K1 + j];
                    }
                    t2sum = group_sum(t, G);
                } else {
                    int nlive = 0;
                    const float sC2 = mufu_sqrt(C2);
                    const uint32_t qx = 0xC0000000u + (uint32_t)qb;  // counters no sample quad uses
                    if (act) {
#pragma unroll 1
                        for (int idx = lig; idx <= nvp; idx += G) {
                            const int j = idx < nvp ? (int)vlist[vs + idx] - p * K : K;
                            const int sl = COMPACT ? sb + idx : sb + j;
                            if (hj[sl] >= 0) {
                                nlive++;
                                t += t2s[sl];
                            } else if (!drop_dead) {
                                if constexpr (NoiseA::kBounded) {
                                    float nz[4];
                                    noise_a.get4(qx, j, gp, nz);
                                    accs[sl] = sC2 * nz[0];
                                }
                            }
                        }
                    }
                    nlive = group_sum_i(nlive, G);
                    t2sum = group_sum(t, G);
                    if (act) {
                        const int n_nl = K1 - nlive;  // logits without per-sample noise
                        const int npad = K - nvp;     // of which masked (they only enter through gzmax)
                        float nz[4] = {0.f, 0.f, 0.f, 0.f};
                        if constexpr (NoiseA::kBounded) {
                            if (!drop_dead) noise_a.get4(qx, K1, gp, nz);
                        }
                        if (lig == 0 && pi.kpad < K) accs[slot_pad] = mufu_sqrt((float)npad * C2) * nz[0];
                        // sum_j sum_s c_s V_sj^2 over those logits: mean n*csum, variance 2 n sum_s c_s^2
                        t2sum += (float)n_nl * csum + mufu_sqrt(2.0f * (float)n_nl * C2) * nz[1];
                    }
                }
            }
            __syncwarp();
        }

        if (!do_finish) {
            // sample-sharded job: publish the partial sums, the caller all-reduces them
            if (act) {
#pragma unroll 1
                for (int j = lig; j < K1; j += G) a.acc[gp * K1 + j] = accs[p * K1 + j];
                if (lig == 0) {
                    a.pixstat[gp * 2 + 0] = t2sum;
                    a.pixstat[gp * 2 + 1] = csum;
                }
            }
        } else {
            // ---- phase 4: chain rule per pixel (SURVEY.md Appendix A.3) ----------------------------------
            const float invSg = a.L.invSg, inv_sr = a.L.inv_sr, invS = a.L.invS;
            const bool from_global = PHASED && !do_sample;
            const bool has_acc = act || (from_global && pvalid);
            if (from_global && pvalid) {
                t2sum = a.pixstat[gp * 2];
                csum = a.pixstat[gp * 2 + 1];
            }
            // grad_zeta_j = acc_j / (S gamma);  gzmax = -sum_j grad_zeta_j over ALL K+1 logits
            float sg = 0.f;
            if (has_acc) {
                if (from_global) {
#pragma unroll 1
                    for (int j = lig; j < K1; j += G) sg += gacc[j] * invSg;
                } else if (!COMPACT && per_sample) {
#pragma unroll 1
                    for (int j = lig; j < K1; j += G) sg += accs[p * K1 + j] * invSg;
                } else {
#pragma unroll 1
                    for (int idx = lig; idx <= nvp; idx += G) {
                        const int j = idx < nvp ? (int)vlist[vs + idx] - p * K : K;
                        sg += accs[COMPACT ? sb + idx : sb + j] * invSg;
                    }
                    if (lig == 0 && pi.kpad < K) sg += accs[slot_pad] * invSg;
                }
            }
            const float gzmax = -group_sum(sg, G);
            if (has_acc && lig == 0) p_gamma += (t2sum - csum) * invSg;
            const float rdenom = __fdividef(1.0f, zf - zn);
            const bool pass = pi.zimax >= pb.eps;
            const float rS = __fdividef(1.0f, (float)pb.S_rast);
            const float* const rsum_t = a.rsum + g0;
            float* const gd_t = a.grad_dists + g0;
            float* const gz_t = a.grad_zbuf + g0;
            float* const gc_t = (a.grad_colors && !fcol) ? a.grad_colors + g0 * 3 : nullptr;
            float* const gfc = fcol ? a.grad_colors : nullptr;  // (num_faces,3), atomic scatter
#pragma unroll 1
            for (int n = vs + lig; n < ve; n += G) {
                const int e = vlist[n];
                const int k = e - p * K;
                const float rsn = rsum_t[e];
                float gz = 0.f;
                const int sl = COMPACT ? sb + (n - vs) : sb + k;
                if (has_acc) gz = (from_global ? gacc[k] : accs[sl]) * invSg;
                const float gzi = gz + ((k == pi.argzi && pass) ? gzmax : 0.f);
                gz_t[e] = -gzi * rdenom;
                const int c = lean ? (int)a.counts[g0 + e] : (int)cnt[n];
                const float pk = (float)c * rS;
                float gP = 0.f;
                if (c != 0) {
                    const float lp = (c == pb.S_rast) ? 0.0f : logf_exact(pk);
                    p_q += lp * gz;        // prod_corrected: inf -> 0 on the scalar side
                    gP = __fdividef(gal * gz, pk);  // log_corrected: 1/0 -> 0
                }
                const float om = 1.0f - pk;
                float excl;
                if (pi.nzero == 0) excl = __fdividef(pi.prod_nz, om);
                else if (pi.nzero == 1) excl = (om == 0.f) ? pi.prod_nz : 0.f;
                else excl = 0.f;
                gP += Gi.w * excl;
                const float gx = gP * (rsn * inv_sr);
                gd_t[e] = -gx;
                p_sigma += gx;
                // grad_colors = w_k * G_rgb
                if (gc_t || gfc) {
                    int h;
                    if (ghist) h = ghist[gp * K1 + k];  // all-shard histogram when sample-sharded
                    else if (act) h = hj[sl];
                    else h = (k == a0) ? sa_loc : 0;
                    if (h > 0) {
                        const float w = (float)h * invS;
                        if (gfc) {
                            float* gc = gfc + 3 * (int)__ldg(p2f_p + k);
                            atomicAdd(gc, w * Gi.x);
                            atomicAdd(gc + 1, w * Gi.y);
                            atomicAdd(gc + 2, w * Gi.z);
                        } else {
                            float* gc = gc_t + e * 3;
                            gc[0] = w * Gi.x;
                            gc[1] = w * Gi.y;
                            gc[2] = w * Gi.z;
                        }
                    }
                }
            }
        }
    }

    // ---- scalar partials of this warp (fixed order) --------------------------------------------------
    if (do_finish) {
        p_sigma = warp_sum(p_sigma);
        p_gamma = warp_sum(p_gamma);
        p_q = warp_sum(p_q);
        if (lane == 0) reinterpret_cast<float4*>(a.partials)[prow] = make_float4(p_sigma, p_gamma, p_q, 0.f);
    }
}

// CTAs (= warps) per SM the main pass is compiled for: 64 registers, no spills; the shared-memory layout allows 30
// (25 / 28 / 32 measured on the sparse set: 0.326 / 0.311 / 0.323 ms)
constexpr int BWD_MAIN_CTAS = 28;
template <class NoiseA, int GT, bool PHASED, bool FACE, bool COMPACT, bool BLOB, int SCORE = 0, bool WOVR = false>
__global__ void __launch_bounds__(FNT, BWD_MAIN_CTAS) shade_bwd_kernel(const BwdArgs a, const NoiseA noise_a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    NoiseA na = noise_a;
    if (a.pb.seed_device) na.mix(__ldg(a.pb.seed_device + 1));  // device-side seed, see shade_fwd.cu
    shade_bwd_tile<NoiseA, GT, PHASED, FACE, COMPACT, BLOB, SCORE, WOVR>(a, na, blockIdx.x, blockIdx.x, smem_raw, threadIdx.x);
}

// Fallback pass of the sparse-first mode (see shade_fwd.cu): work-list tiles as half-size tiles with dense
// per-logit arrays; their scalar partials go to the rows after the main pass's.
template <class NoiseA, int GT, bool FACE>
__global__ void __launch_bounds__(FBT, 12) shade_bwd_fallback_kernel(const BwdArgs a, const NoiseA noise_a, int64_t prow0) {
    extern __shared__ __align__(16) unsigned char smem_all[];
    unsigned char* smem_raw = smem_all + (threadIdx.x >> 5) * a.L.warp_smem;  // FBT/32 independent warps per CTA
    const int n = 2 * a.worklist[0];
    NoiseA na = noise_a;
    if (a.pb.seed_device) na.mix(__ldg(a.pb.seed_device + 1));
#pragma unroll 1
    for (;;) {  // persistent warps fetch half-tiles dynamically
        int i = 0;
        if ((threadIdx.x & 31) == 0) i = n > 0 ? atomicAdd(a.worklist + 1, 1) : 0;
        i = __shfl_sync(FULL, i, 0);
        if (i >= n) break;
        const int64_t tile = (int64_t)a.worklist[4 + (i >> 1)] * 2 + (i & 1);
        if (tile < a.L.ntiles) {
            shade_bwd_tile<NoiseA, GT, false, FACE, false, false>(a, na, tile, prow0 + i, smem_raw, threadIdx.x & 31);
        } else if ((threadIdx.x & 31) == 0) {
            reinterpret_cast<float4*>(a.partials)[prow0 + i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncwarp();
    }
}

// deterministic final reduction of the per-tile scalar partials (one CTA)
//   out[0] = d/dsigma = sum gx                         (smoothrast.py:57-58)
//   out[1] = d/dgamma = score term + q/alpha           (smoothagg.py:72 and :329-332 through gamma/alpha)
//   out[2] = d/dalpha = -q gamma / alpha^2
__global__ void __launch_bounds__(1024) finalize_scalars_kernel(const float* partials, int64_t n, const int32_t* worklist,
                                                                float gamma, float alpha, float* out) {
    __shared__ double red[3][32];
    if (worklist) n += 2 * (int64_t)worklist[0];  // rows of the fallback pass
    double s0 = 0, s1 = 0, s2 = 0;
    // eight independent loads in flight per thread (one CTA walks every row: the loop is latency-bound otherwise);
    // a thread still adds its rows in increasing order, so the result does not depend on the unrolling
    const float4* const rows = reinterpret_cast<const float4*>(partials);
    int64_t t = threadIdx.x;
    for (; t + 7 * 1024 < n; t += 8 * 1024) {
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = __ldg(rows + t + u * 1024);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            s0 += v[u].x;
            s1 += v[u].y;
            s2 += v[u].z;
        }
    }
    for (; t < n; t += 1024) {
        const float4 v = __ldg(rows + t);
        s0 += v.x;
        s1 += v.y;
        s2 += v.z;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s0 += __shfl_xor_sync(FULL, s0, o);
        s1 += __shfl_xor_sync(FULL, s1, o);
        s2 += __shfl_xor_sync(FULL, s2, o);
    }
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = s0;
        red[1][threadIdx.x >> 5] = s1;
        red[2][threadIdx.x >> 5] = s2;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double r0 = 0, r1 = 0, q = 0;
        for (int w = 0; w < 32; ++w) {
            r0 += red[0][w];
            r1 += red[1][w];
            q += red[2][w];
        }
        out[0] = (float)r0;
        out[1] = (float)(r1 + q / (double)alpha);
        out[2] = (float)(-q * (double)gamma / ((double)alpha * (double)alpha));
    }
}

template <class K>
static int set_smem(K kern, size_t smem) {
    if (smem > 48 * 1024) return (int)cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    return 0;
}

template <class NA, int GT, bool PHASED, bool FACE, bool COMPACT, bool BLOB = false, int SCORE = 0, bool WOVR = false>
static int launch_bwd_f(const BwdArgs& a, const NA& na, cudaStream_t st) {
    const size_t smem = (size_t)a.L.warp_smem;
    if (int rc = set_smem(shade_bwd_kernel<NA, GT, PHASED, FACE, COMPACT, BLOB, SCORE, WOVR>, smem)) return rc;
    shade_bwd_kernel<NA, GT, PHASED, FACE, COMPACT, BLOB, SCORE, WOVR><<<(unsigned)a.L.ntiles, FNT, smem, st>>>(a, na);
    return (int)cudaGetLastError();
}
template <class NA, int GT, bool PHASED, int SCORE = 0, bool WOVR = false>
static int launch_bwd_t(const BwdArgs& a, const NA& na, cudaStream_t st) {
    return a.pb.face_colors ? launch_bwd_f<NA, GT, PHASED, true, false, false, SCORE, WOVR>(a, na, st)
                            : launch_bwd_f<NA, GT, PHASED, false, false, false, SCORE, WOVR>(a, na, st);
}
// sparse-first main pass (compact per-logit arrays); PN = the Philox variant
template <class PN, int GT>
static int launch_bwd_c(const BwdArgs& a, const PN& na, cudaStream_t st) {
    if (a.blob) {  // forward left tile blobs: no re-scan, no logit recomputation (the common geometries only)
        if constexpr (GT == 2 || GT == 4) {
            return a.pb.face_colors ? launch_bwd_f<PN, GT, false, true, true, true>(a, na, st)
                                    : launch_bwd_f<PN, GT, false, false, true, true>(a, na, st);
        }
    }
    return a.pb.face_colors ? launch_bwd_f<PN, GT, false, true, true>(a, na, st)
                            : launch_bwd_f<PN, GT, false, false, true>(a, na, st);
}
template <class PN, int GT, bool FACE>
static int launch_bwd_fb(const BwdArgs& a, const PN& na, int64_t prow0, cudaStream_t st) {
    const size_t smem = (size_t)a.L.warp_smem * (FBT / 32);
    if (int rc = set_smem(shade_bwd_fallback_kernel<PN, GT, FACE>, smem)) return rc;
    shade_bwd_fallback_kernel<PN, GT, FACE><<<resident_grid(shade_bwd_fallback_kernel<PN, GT, FACE>, FBT, smem), FBT, smem, st>>>(a, na, prow0);
    return (int)cudaGetLastError();
}

// both phases in one launch, in-kernel noise
template <class PN>
static int launch_bwd_production(const BwdArgs& a, const BwdArgs* fb, cudaStream_t st) {
    const PN pa(a.pb.seed_agg, 1, a.pb.pixel_offset);
    int rc;
    if (fb) {  // sparse-first: compact main pass, then half-size tiles for whatever did not fit
        switch (a.L.G) {
            case 1: rc = launch_bwd_c<PN, 1>(a, pa, st); break;
            case 2: rc = launch_bwd_c<PN, 2>(a, pa, st); break;
            case 4: rc = launch_bwd_c<PN, 4>(a, pa, st); break;
            default: rc = launch_bwd_c<PN, 8>(a, pa, st); break;
        }
        if (rc) return rc;
        const bool face = a.pb.face_colors != nullptr;
        switch (fb->L.G) {
            case 2: return face ? launch_bwd_fb<PN, 2, true>(*fb, pa, a.L.ntiles, st) : launch_bwd_fb<PN, 2, false>(*fb, pa, a.L.ntiles, st);
            case 4: return face ? launch_bwd_fb<PN, 4, true>(*fb, pa, a.L.ntiles, st) : launch_bwd_fb<PN, 4, false>(*fb, pa, a.L.ntiles, st);
            case 8: return face ? launch_bwd_fb<PN, 8, true>(*fb, pa, a.L.ntiles, st) : launch_bwd_fb<PN, 8, false>(*fb, pa, a.L.ntiles, st);
            default: return face ? launch_bwd_fb<PN, 16, true>(*fb, pa, a.L.ntiles, st) : launch_bwd_fb<PN, 16, false>(*fb, pa, a.L.ntiles, st);
        }
    }
    switch (a.L.G) {  // lanes per pixel known at compile time
        case 1: return launch_bwd_t<PN, 1, false>(a, pa, st);
        case 2: return launch_bwd_t<PN, 2, false>(a, pa, st);
        case 4: return launch_bwd_t<PN, 4, false>(a, pa, st);
        default: return launch_bwd_t<PN, 8, false>(a, pa, st);
    }
}

int launch_shade_bwd(const BwdArgs& a, const BwdArgs* fb, float* grad_scalars, cudaStream_t st) {
    int rc;
    const uint32_t both = PERT_PH_BWD_SAMPLE | PERT_PH_BWD_FINISH;
    const bool phased = (a.pb.flags & both) != both || a.hist != nullptr;
    if (a.pb.flags & PERT_F_CAUCHY) {  // Cauchy pair: the dense phase-capable instantiation, as forward (shade_fwd.cu)
        if (a.pb.noise_agg) {
            ExplicitNoise xa{a.pb.noise_agg, a.L.P, a.pb.K + 1, a.pb.S_agg};
            rc = launch_bwd_t<ExplicitNoise, 0, true, 1>(a, xa, st);
        } else {
            rc = launch_bwd_t<PhiloxCauchy, 0, true, 1>(a, PhiloxCauchy(a.pb.seed_agg, 1, a.pb.pixel_offset), st);
        }
    } else if (a.pb.flags & PERT_F_NO_VR) {  // no control variates: the same dense instantiation, Gaussian noise
        if (a.pb.noise_agg) {
            ExplicitNoise xa{a.pb.noise_agg, a.L.P, a.pb.K + 1, a.pb.S_agg};
            rc = launch_bwd_t<ExplicitNoise, 0, true, 0, true>(a, xa, st);
        } else {
            rc = launch_bwd_t<PhiloxNoise, 0, true, 0, true>(a, PhiloxNoise(a.pb.seed_agg, 1, a.pb.pixel_offset), st);
        }
    } else if (a.pb.noise_agg) {
        ExplicitNoise xa{a.pb.noise_agg, a.L.P, a.pb.K + 1, a.pb.S_agg};
        rc = launch_bwd_t<ExplicitNoise, 0, true>(a, xa, st);
    } else if (phased) {  // sample-sharded job: compile-time lanes per pixel for the benchmark geometries
        PhiloxNoise pa(a.pb.seed_agg, 1, a.pb.pixel_offset);
        switch (a.L.G) {
            case 4: rc = launch_bwd_t<PhiloxNoise, 4, true>(a, pa, st); break;
            case 8: rc = launch_bwd_t<PhiloxNoise, 8, true>(a, pa, st); break;
            default: rc = launch_bwd_t<PhiloxNoise, 0, true>(a, pa, st); break;
        }
    } else {
        rc = (a.pb.flags & PERT_F_PHILOX7) ? launch_bwd_production<PhiloxNoise7>(a, fb, st)
                                           : launch_bwd_production<PhiloxNoise>(a, fb, st);
    }
    if (rc) return rc;
    if (a.pb.flags & PERT_PH_BWD_FINISH) {
        finalize_scalars_kernel<<<1, 1024, 0, st>>>(a.partials, a.L.ntiles, fb ? a.worklist : nullptr, a.pb.gamma,
                                                    a.pb.alpha, grad_scalars);
        return (int)cudaGetLastError();
    }
    return 0;
}

}  // namespace pert
