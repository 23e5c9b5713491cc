// Fused forward of the perturbed shader (pert_shade_fwd in include/pertshade.h).
//
// Reference path: smooth_rgb_blend (randomras/random_rasterizer.py:34-56) -> randomHeaviside.forward
// (randomras/smoothrast.py:15-37) -> GaussianAgg.aggregate (randomras/smoothagg.py:196-205) ->
// randomArgmax.forward (randomras/smoothagg.py:13-42) -> blend.
//
// One warp (= one CTA) per tile of tp pixels, no block-level synchronisation.  Phases of a tile:
//   0  scan pix_to_face (128-bit loads) -> compact list of valid entries; zbuf/dists only for those
//   1  coverage samples of the entries whose sign can flip (Philox in registers) -> counts, rsum
//   2  per-pixel logits (G lanes per pixel), list of logits that can win a sample
//   3  perturbed argmax samples over (pixel, sample-quad) items -> winners, histogram
//   4  blend -> image; per-pixel state (a0, active) for backward
#include "kernels.h"
#include "tile.cuh"

namespace pert {

int fwd_smem_layout(int tp, int cap, SmemLayout& L) {
    Carver cv(L);
    cv.take(cap, 2);       // vlist
    cv.take(cap + tp, 4);  // xs | lz
    cv.take(cap, 2);       // cnt
    cv.take(cap + tp, 4);  // rs | hl
    cv.take(cap + tp, 2);  // rlist | lj
    cv.take(64, 2);        // ring (compound sampler)
    const int rast_bytes = L.bytes;
    cv.take(cap, 4);       // zs: from here on, arrays the coverage-sample launch of a split pass never touches
    cv.take(tp + 1, 4);    // vstart
    cv.take(tp, 4);        // pinfo
    cv.take(tp, 2);        // plist
    return rast_bytes;
}

// Main pass of the sparse-first mode: a tile with at least this many entries for the compound sampler goes to the fallback
// pass.  Elsewhere, fewer compound entries than kCmpMin in a tile are drawn by the per-sample loop instead.
constexpr int kDeferMin = 48;
constexpr int kCmpMin = 12;

// GT = lanes per pixel as a compile-time constant (1, 2, 4, 8), or 0 to read it from the launch record.
// PHASED = false is the production instantiation: all three phases in one launch, no global histogram
// (the phase-split code of the sample-sharded job is compiled out, which keeps the hot code small: the
// kernel is instruction-fetch sensitive, every warp walks the whole body once per tile).
// DEFER = true (main pass of the sparse-first mode): a tile with enough entries for the compound coverage sampler is
// handed to the fallback pass like a tile that overflows the compact arrays, so that this instantiation carries no
// compound-sampler code at all (the kernel is instruction-fetch bound on sparse fragments: every instruction of a
// path it rarely takes costs the common path)
// CPH = the phases this instantiation carries when PHASED is false (PERT_PH_* bits; all of them by default).  The
// fallback pass runs as two launches, coverage samples (CPH = RAST: counts / rsum go to global memory, where backward
// wants them anyway) and then aggregation + blend (CPH = AGG | BLEND: reads the counts back), because one kernel with
// both exceeds the 32 KB instruction cache of an SM and every warp walks the whole body once per tile.
// SCORE = the score of the coverage noise in rsum (philox.cuh noise_score): 0 Gaussian, 1 Cauchy.
// WOVR = true: the estimator without control variates (PERT_F_NO_VR): rsum = sum_s h psi(U), so an entry that is
// covered by every sample still draws them all; only the side x < -sigma*Umax (h = 0 always) is skipped, and the
// compound sampler (which produces sum_s (h - h0) U only) is compiled out.  Counts, winners and image are unchanged.
// RENDER = true: the forward-only render (pert_shade_render, pert_shade_render_phase): nothing is stored for backward (no
// rsum, winners, pixstate or tile blob); coverage computes counts only, from the same counters, so counts, histogram and
// image are those of the training forward.  Counts go to global memory only in a coverage-only call: the coverage-sample
// launch of a split fallback pass (a.counts is then the caller's S-independent workspace), which the aggregation launch
// reads back, or the RAST call of a phase-split render (PHASED).
// Fallback records (common.cuh; training with a tile blob, a.blob then points at the records region): the coverage launch
// stores the half-tile's valid list; REC = true (aggregation launch) loads it instead of re-scanning pix_to_face and stores
// what backward would recompute, the per-pixel logit summary and zeta.
template <class NoiseR, class NoiseA, int GT, bool PHASED, bool DEFER = false, int CPH = 0x70, int SCORE = 0,
          bool WOVR = false, bool RENDER = false, bool REC = false>
__device__ __forceinline__ void shade_fwd_tile(const FwdArgs& a, const NoiseR& noise_r, const NoiseA& noise_a,
                                               const int64_t tile, unsigned char* smem_raw, const int lane) {
    const pert_problem& pb = a.pb;
    const int G = GT ? GT : a.L.G;
    const int gshift = GT ? (GT == 16 ? 4 : GT == 8 ? 3 : GT == 4 ? 2 : GT == 2 ? 1 : 0) : a.L.gshift;
    const int K = pb.K, K1 = K + 1, tp = 32 >> gshift;
    const int64_t pix0 = tile * tp;
    const int npx = (int)min((int64_t)tp, a.L.P - pix0);
    const int E = npx * K;
    const int64_t g0 = pix0 * K;
    const uint32_t flags = pb.flags;
    const bool do_rast = PHASED ? (flags & PERT_PH_RAST) != 0 : (CPH & PERT_PH_RAST) != 0,
               do_agg = PHASED ? (flags & PERT_PH_AGG) != 0 : (CPH & PERT_PH_AGG) != 0,
               do_blend = PHASED ? (flags & PERT_PH_BLEND) != 0 : (CPH & PERT_PH_BLEND) != 0;
    int32_t* const ghist = PHASED ? a.hist : nullptr;
    const float* const zbuf_t = pb.zbuf + g0;
    const float* const dists_t = pb.dists + g0;
    uint16_t* const counts_t = a.counts + g0;
    float* const rsum_t = a.rsum + g0;
    const bool no_skip = flags & PERT_F_NO_SKIP;
    const int p = lane >> gshift, lig = lane & (G - 1);
    const bool pvalid = p < npx;
    const int64_t gp = pix0 + p;
    const unsigned lt = (1u << lane) - 1u;

    Taker cv(smem_raw, a.L.sm);  // layout: fwd_smem_layout (every array is compact: `cap` valid entries)
    uint16_t* vlist = cv.take<uint16_t>();
    float* xs = cv.take<float>();          // x = -dists (compact); later lz: logits of the live list
    uint16_t* cnt = cv.take<uint16_t>();
    float* rs = cv.take<float>();          // sum_s (h-h0) U (compact); later hl: histogram of the live list
    uint16_t* rlist = cv.take<uint16_t>();  // entries that need coverage samples; later lj: live logit ids
    uint16_t* ring = cv.take<uint16_t>();
    float* zs = cv.take<float>();          // zbuf -> zi -> zeta (compact)
    int* vstart = cv.take<int>();
    int* pinfo = cv.take<int>();  // nlive | a0l << 16 of every pixel
    uint16_t* plist = cv.take<uint16_t>();
    const int cap = a.L.cap;
    float* lz = xs;
    int* hl = reinterpret_cast<int*>(rs);
    uint16_t* lj = rlist;
    // this tile's blob (main pass) or record (fallback pass) in a.blob; derived where used, so that no pointer stays live
    auto blob_of = [&]() { return a.blob + tile * (int64_t)(CPH == 0x70 ? blob_words(tp, cap) : fbrec_words(tp, cap)); };

    // ---- phase 0 -----------------------------------------------------------------------------------
    int nv;
    if constexpr (REC) {
        const int32_t* const bl = blob_of();
        nv = __ldg(bl);
        const int32_t* const src = bl + blob_vlist_off(tp);
#pragma unroll 1
        for (int i = lane; i < ((nv + 1) >> 1); i += 32) reinterpret_cast<int32_t*>(vlist)[i] = __ldg(src + i);
    } else {
        nv = scan_valid(pb.pix_to_face + g0, E, a.L.vec_ok, vlist, cap);
    }
    const int sa_loc = a.L.sa_loc;
    if (nv > cap) {
        // sparse-first mode: this tile has more valid entries than the compact arrays hold: hand it to the
        // fallback pass (half-size tiles, full capacity)
        if (lane == 0) {
            a.worklist[4 + atomicAdd(a.worklist, 1)] = (int32_t)tile;
            if (a.blob) blob_of()[0] = -1;
        }
        return;
    }
    if (nv == 0) {
        // nothing but padding: background, alpha 0, every sample picks the background (index K)
        if (do_agg && ghist) {
#pragma unroll 1
            for (int i = lane; i < npx * K1; i += 32) ghist[pix0 * K1 + i] = ((i % K1) == K) ? sa_loc : 0;
        }
        if (!RENDER && do_agg && lane < npx) a.pixstate[pix0 + lane] = (uint16_t)K;
        if (!PHASED && !RENDER && !REC && a.blob && lane == 0) blob_of()[0] = 0;
        if (do_blend && lane < npx)
            reinterpret_cast<float4*>(a.image)[pix0 + lane] =
                make_float4(pb.background[0], pb.background[1], pb.background[2], 0.0f);
        return;
    }
    __syncwarp();
    if constexpr (CPH == (int)PERT_PH_RAST && !RENDER) {
        if (a.blob) {  // the valid list, for the aggregation launch and backward
            int32_t* const bl = blob_of();
            if (lane == 0) bl[0] = nv;
#pragma unroll 1
            for (int i = lane; i < ((nv + 1) >> 1); i += 32)
                bl[blob_vlist_off(tp) + i] = reinterpret_cast<const int32_t*>(vlist)[i];
        }
    }
    if (do_agg || do_blend) pixel_ranges(vlist, nv, K, tp, vstart);

    // ---- phase 1: stage valid entries, coverage samples ---------------------------------------------
    const int sr_loc = pb.s_rast_end - pb.s_rast_begin;
    const float thr = (NoiseR::kBounded && !no_skip) ? pb.sigma * kNoiseAbsMax * 1.0001f : CUDART_INF_F;
    // compound sampler (tile.cuh) for the entries with |x| >= x_cmp: the default with in-kernel noise
    const bool compound = !WOVR && NoiseR::kBounded && !no_skip && !(flags & PERT_F_PER_SAMPLE_NOISE);
    const float x_cmp = compound ? a.L.t_compound * pb.sigma : CUDART_INF_F;
    uint16_t* const blist = rlist + cap - 1;  // stored downwards: the two lists share one array of cap entries
    int nlist = 0, nblist = 0;
#pragma unroll 1
    for (int n0 = 0; n0 < nv; n0 += 32) {
        const int n = n0 + lane;
        bool need = false, cmp = false;
        if (n < nv) {
            const int e = vlist[n];
            if (do_agg || do_blend) {
                zs[n] = __ldg(zbuf_t + e);
                if (!pb.face_colors) prefetch_l1(pb.colors + (g0 + e) * 3);  // blended at the very end of the tile
            }
            if (do_rast) {
                const float x = -__ldg(dists_t + e);
                xs[n] = x;
                // |x| beyond the largest possible sigma*|U| cannot flip: exact, not an approximation
                need = WOVR ? x >= -thr : fabsf(x) <= thr;
                cmp = need && fabsf(x) >= x_cmp;
                if (!need) {
                    cnt[n] = (x >= 0.0f) ? (uint16_t)sr_loc : (uint16_t)0;
                    if constexpr (!RENDER) rs[n] = 0.0f;
                }
            } else {
                cnt[n] = counts_t[e];
            }
        }
        if (do_rast) {
            if constexpr (DEFER) {  // one list; the tile is handed over if enough of it is worth the compound sampler
                const unsigned b = __ballot_sync(FULL, need);
                if (need) rlist[nlist + __popc(b & lt)] = (uint16_t)n;
                nlist += __popc(b);
                nblist += __popc(__ballot_sync(FULL, cmp));
            } else {
                const unsigned b = __ballot_sync(FULL, need && !cmp), bc = __ballot_sync(FULL, cmp);
                if (need && !cmp) rlist[nlist + __popc(b & lt)] = (uint16_t)n;
                if (cmp) blist[-(nblist + __popc(bc & lt))] = (uint16_t)n;
                nlist += __popc(b);
                nblist += __popc(bc);
            }
        }
    }
    __syncwarp();
    if (do_rast) {
        if constexpr (DEFER) {
            if (nblist >= kDeferMin) {
                if (lane == 0) {
                    a.worklist[4 + atomicAdd(a.worklist, 1)] = (int32_t)tile;
                    if (a.blob) blob_of()[0] = -1;
                }
                return;
            }
        }
        if (!DEFER && nblist > 0 && nblist < kCmpMin) {
            // a handful of entries: the per-sample loop spreads each entry's samples over the idle lanes, which beats
            // one lane per entry (the lists share one array: the moved entries are read before they can be overwritten)
            const int moved = lane < nblist ? blist[-lane] : 0;
            __syncwarp();
            if (lane < nblist) rlist[nlist + lane] = (uint16_t)moved;
            nlist += nblist;
            nblist = 0;
            __syncwarp();
        }
        if constexpr (NoiseR::kBounded && !DEFER && !WOVR) {
            if (nblist > 0) {
                const CompoundCtx<NoiseR> cc{noise_r, vlist, xs, cnt, rs, K, a.L.invK, pix0, a.L.inv_sigma, sr_loc,
                                             0x40000000u + 2u * (uint32_t)(pb.s_rast_begin >> 2)};
                if constexpr (RENDER)
                    rast_compound_count_list(cc, blist, nblist, a.L.t_bucket[0] * pb.sigma, a.L.t_bucket[1] * pb.sigma, ring);
                else
                    rast_compound_list(cc, blist, nblist, a.L.t_bucket[0] * pb.sigma, a.L.t_bucket[1] * pb.sigma, ring);
            }
        }
        rast_sample_list<NoiseR, SCORE, WOVR, RENDER>(noise_r, rlist, nlist, vlist, xs, cnt, rs, K, a.L.invK, pix0, pb.sigma, a.L.inv_sigma, pb.s_rast_begin,
                         pb.s_rast_end, !no_skip, a.L.lpe_r);
        __syncwarp();
        if (!RENDER || !do_agg) {
#pragma unroll 1
            for (int n = lane; n < nv; n += 32) {
                const int e = vlist[n];
                counts_t[e] = cnt[n];
                if constexpr (!RENDER) rsum_t[e] = rs[n];
            }
        }
    }
    if (!do_agg && !do_blend) return;
    __syncwarp();

    // ---- phase 2: logits, alpha, live lists ---------------------------------------------------------
    const float gal = a.L.gal;  // gamma / alpha as an fp32 scalar division (smoothagg.py:201), done on the host
    float zn = 1.0f, zf = 100.0f;
    if (pvalid) {
        const int b = pb.depth_len > 1 ? batch_of(pix0, p, a.L.HW) : 0;
        zn = __ldg(pb.znear + b);
        zf = __ldg(pb.zfar + b);
    }
    const PixPrep pi = prep_pixels(p, lig, G, pvalid, K, vstart, vlist, cnt, zs, zn, zf, pb.S_rast, gal, pb.eps);
    const float px_alpha = 1.0f - (pi.nzero ? 0.0f : pi.prod_nz);
    const int vs = pvalid ? vstart[p] : 0, ve = pvalid ? vstart[p + 1] : 0;
    const int nvp = ve - vs;
    const int lb = vs + p;  // this pixel's slots in lz / lj / hl: nvp + 1 of them
    int nlive = 0, a0l = 0;
    bool active = false;
    __syncwarp();
    if (do_agg) {
        // a logit can win some sample only if zeta_j + gamma*Umax >= zeta_max - gamma*Umax
        const float floor_v = pi.zeta_max - live_cut(pb.gamma, pi.zeta_max, NoiseA::kBounded && !no_skip);
        const int iters = warp_max_i((nvp + G) / G);  // ceil((nvp + 1) / G), uniform for the ballots
        const unsigned gmask = (G == 32) ? FULL : ((1u << G) - 1u);
        const int gsh = p * G;
#pragma unroll 1
        for (int it = 0; it < iters; ++it) {
            const int idx = it * G + lig;
            float z = -CUDART_INF_F;
            int j = K;
            if (pvalid && idx < nvp) {
                z = zs[vs + idx];
                j = (int)vlist[vs + idx] - p * K;
            } else if (pvalid && idx == nvp) {
                z = pi.zbg;
            }
            const bool lv = z > -CUDART_INF_F && z >= floor_v;
            const unsigned gb = (__ballot_sync(FULL, lv) >> gsh) & gmask;
            if (lv) {
                const int pos = lb + nlive + __popc(gb & ((1u << lig) - 1u));
                lz[pos] = z;
                lj[pos] = (uint16_t)j;
                hl[pos] = 0;
            }
            const unsigned a0b = (__ballot_sync(FULL, lv && j == pi.a0) >> gsh) & gmask;
            if (a0b) a0l = nlive + __popc(gb & ((1u << (__ffs(a0b) - 1)) - 1u));
            nlive += __popc(gb);
        }
        __syncwarp();

        // ---- phase 3: perturbed argmax samples (smoothagg.py:33-36) ---------------------------------
        const bool multi = pvalid && lig == 0 && nlive > 1;
        const unsigned mb = __ballot_sync(FULL, multi);
        if (multi) plist[__popc(mb & lt)] = (uint16_t)p;
        if (pvalid && lig == 0) pinfo[p] = nlive | (a0l << 16);
        const int np = __popc(mb);
        __syncwarp();
        if (np > 2) {
            // order the listed pixels by their number of live logits: the pixels that share a warp pass then
            // loop about equally long (less divergence)
            const int myp = lane < np ? plist[lane] : 0;
            const int myn = lane < np ? (pinfo[myp] & 0xffff) : -1;
            int rank = 0;
#pragma unroll 1
            for (int i = 0; i < np; ++i) {
                const int on = __shfl_sync(FULL, myn, i);
                rank += (on > myn || (on == myn && i < lane)) ? 1 : 0;
            }
            __syncwarp();
            if (lane < np) plist[rank] = (uint16_t)myp;
            __syncwarp();
        }
        if (np > 0) {
            const int qb = pb.s_agg_begin >> 2, qe = (pb.s_agg_end + 3) >> 2;
            const int lpe = a.L.lpe_a;
            const int gpw = 32 >> a.L.lpe_a_shift;
            const int lq = lane & (lpe - 1);
            const float gamma = pb.gamma;
            const bool pack = a.L.win_bytes == 1 && (sa_loc & 3) == 0;
#pragma unroll 1
            for (int base = 0; base < np; base += gpw) {
                const int pe = base + (lane >> a.L.lpe_a_shift);
                if (pe >= np) continue;
                const int pp = plist[pe];
                const int plb = vstart[pp] + pp;
                const int pn = pinfo[pp] & 0xffff, pa0 = pinfo[pp] >> 16;
                const int64_t pgp = pix0 + pp;
#pragma unroll 1
                for (int q = qb + lq; q < qe; q += lpe) {
                    float best[4] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
                    int bi[4] = {0, 0, 0, 0};
#pragma unroll 1
                    for (int l = 0; l < pn; ++l) {
                        const int j = lj[plb + l];
                        const float z = lz[plb + l];
                        float nz[4];
                        noise_a.get4(q, j, pgp, nz);
#pragma unroll
                        for (int t = 0; t < 4; ++t) {
                            const float v = __fadd_rn(z, __fmul_rn(gamma, nz[t]));
                            if (v > best[t]) {
                                best[t] = v;
                                bi[t] = l;
                            }
                        }
                    }
                    int wj[4];
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        wj[t] = lj[plb + bi[t]];
                        const int s = q * 4 + t;
                        if (s >= pb.s_agg_begin && s < pb.s_agg_end && bi[t] != pa0) atomicAdd(&hl[plb + bi[t]], 1);
                    }
                    if constexpr (RENDER) continue;  // the histogram stays on chip; no winners
                    const int s0 = q * 4 - pb.s_agg_begin;
                    if (pack && q * 4 + 3 < pb.s_agg_end) {
                        reinterpret_cast<uint32_t*>(a.winners)[(pgp * sa_loc + s0) >> 2] =
                            (uint32_t)wj[0] | ((uint32_t)wj[1] << 8) | ((uint32_t)wj[2] << 16) | ((uint32_t)wj[3] << 24);
                    } else {
#pragma unroll
                        for (int t = 0; t < 4; ++t)
                            if (q * 4 + t < pb.s_agg_end) store_winner(a.winners, a.L.win_bytes, pgp * sa_loc + s0 + t, wj[t]);
                    }
                }
            }
        }
        __syncwarp();
        // histogram of the unperturbed winner = all the samples nobody else won
        int others = 0;
#pragma unroll 1
        for (int l = lig; l < nlive; l += G)
            if (l != a0l) others += hl[lb + l];
        others = group_sum_i(others, G);
        active = others > 0;
        if (pvalid && lig == 0) {
            hl[lb + a0l] = sa_loc - others;
            if constexpr (!RENDER) a.pixstate[gp] = (uint16_t)(pi.a0 | (active ? 0x8000 : 0));
        }
        if (!PHASED && !RENDER && (CPH == 0x70 || REC) && a.blob) {
            // what backward would recompute from pix_to_face / zbuf / counts (layout: common.cuh); a fallback record already
            // holds nv and the valid list (coverage launch) and carries no counts
            int32_t* const bl = blob_of();
            if (CPH == 0x70 && lane == 0) bl[0] = nv;
            for (int i = lane; i <= tp; i += 32) bl[1 + i] = i <= npx ? vstart[i] : nv;
            if (pvalid && lig == 0) {
                int32_t* const bp = bl + blob_pix_off(tp) + 6 * p;
                bp[0] = __float_as_int(pi.zmax);
                bp[1] = __float_as_int(pi.zimax);
                bp[2] = __float_as_int(pi.prod_nz);
                bp[3] = __float_as_int(pi.zeta_max);
                bp[4] = pi.argzi | (pi.a0 << 16);
                bp[5] = pi.nzero | (pi.kpad << 16);
            }
            if constexpr (CPH == 0x70) {
                const uint32_t* const vl32 = reinterpret_cast<const uint32_t*>(vlist);
                const uint32_t* const cn32 = reinterpret_cast<const uint32_t*>(cnt);
                const int nw = (nv + 1) >> 1;
#pragma unroll 1
                for (int i = lane; i < nw; i += 32) {
                    bl[blob_vlist_off(tp) + i] = (int32_t)vl32[i];
                    bl[blob_cnt_off(tp, cap) + i] = (int32_t)cn32[i];
                }
            }
            const int zoff = CPH == 0x70 ? blob_zeta_off(tp, cap) : fbrec_zeta_off(tp, cap);
#pragma unroll 1
            for (int i = lane; i < nv; i += 32) bl[zoff + i] = __float_as_int(zs[i]);
        }
        __syncwarp();
        if (ghist) {
            // dense (P,K1) histogram for the sample-sharded job: zeros, then the live entries
#pragma unroll 1
            for (int i = lane; i < npx * K1; i += 32) ghist[pix0 * K1 + i] = 0;
            __syncwarp();
#pragma unroll 1
            for (int l = lig; l < nlive; l += G) ghist[gp * K1 + lj[lb + l]] = hl[lb + l];
        }
    }
    if (!do_blend) return;

    // ---- phase 4: blend (random_rasterizer.py:50-54) ------------------------------------------------
    float r = 0.f, g = 0.f, bl = 0.f;
    const float fS = (float)pb.S_agg;
    const float* const colors_p = pb.colors + gp * K * 3;
    const float* const fcol = pb.face_colors;  // per-face colours gathered through pix_to_face, or NULL
    const int64_t* const p2f_p = pb.pix_to_face + gp * K;
    if (do_agg) {
#pragma unroll 1
        for (int l = lig; l < nlive; l += G) {
            const int hcount = hl[lb + l];
            if (hcount > 0) {
                const float w = (float)hcount / fS;
                const int j = lj[lb + l];
                if (j < K) {
                    const float* c = fcol ? fcol + 3 * (int)__ldg(p2f_p + j) : colors_p + j * 3;
                    r += w * __ldg(c);
                    g += w * __ldg(c + 1);
                    bl += w * __ldg(c + 2);
                } else {
                    r += w * pb.background[0];
                    g += w * pb.background[1];
                    bl += w * pb.background[2];
                }
            }
        }
    } else if (PHASED) {
        // histogram summed over all sample shards (read from global memory)
        const int32_t* hg = ghist + gp * K1;
#pragma unroll 1
        for (int idx = lig; idx <= nvp && pvalid; idx += G) {
            const int j = idx < nvp ? (int)vlist[vs + idx] - p * K : K;
            const int hcount = hg[j];
            if (hcount > 0) {
                const float w = (float)hcount / fS;
                if (j < K) {
                    const float* c = fcol ? fcol + 3 * (int)__ldg(p2f_p + j) : colors_p + j * 3;
                    r += w * __ldg(c);
                    g += w * __ldg(c + 1);
                    bl += w * __ldg(c + 2);
                } else {
                    r += w * pb.background[0];
                    g += w * pb.background[1];
                    bl += w * pb.background[2];
                }
            }
        }
    }
    r = group_sum(r, G);
    g = group_sum(g, G);
    bl = group_sum(bl, G);
    if (pvalid && lig == 0) reinterpret_cast<float4*>(a.image)[gp] = make_float4(r, g, bl, px_alpha);
}

// CTAs (= warps) per SM of the main kernel.  Training: 32 (64 registers); the Cauchy instantiations (SCORE = 1) and those
// without control variates (WOVR) get 24 (80 registers): at 64 the in-kernel Cauchy stream and the ungated coverage samples
// of WOVR spill.  Render: 28 (72 registers; at 64 the Philox-10 and explicit-noise renders spill), 24 for Cauchy and for the
// phase-split render (its in-kernel Gaussian and explicit-rast instantiations spill at 72).
constexpr int fwd_min_ctas(int score, bool wovr, bool render, bool phased) {
    return (score || wovr || (render && phased)) ? 24 : render ? 28 : 32;
}

template <class NoiseR, class NoiseA, int GT, bool PHASED, bool DEFER, int SCORE, bool WOVR, bool RENDER>
__global__ void __launch_bounds__(FNT, fwd_min_ctas(SCORE, WOVR, RENDER, PHASED))
    shade_fwd_kernel(const FwdArgs a, const NoiseR noise_r, const NoiseA noise_a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    NoiseR nr = noise_r;
    NoiseA na = noise_a;
    if (a.pb.seed_device) {  // seeds that live on the device: a captured CUDA graph draws fresh noise at every replay
        nr.mix(__ldg(a.pb.seed_device));
        na.mix(__ldg(a.pb.seed_device + 1));
    }
    shade_fwd_tile<NoiseR, NoiseA, GT, PHASED, DEFER, 0x70, SCORE, WOVR, RENDER>(a, nr, na, blockIdx.x, smem_raw, threadIdx.x);
}

// Fallback pass of the sparse-first mode: the tiles whose valid entries did not fit the compact arrays,
// as half-size tiles (GT lanes per pixel = twice the main pass's) with full capacity.  Few persistent CTAs
// walk the work list; it is empty for sparse (real) fragments.  Two launches, CPH = RAST and CPH = AGG | BLEND (see
// shade_fwd_tile); with a tile blob the second one reads the valid lists the first one stored (REC).
// CTAs per SM of the fallback launches: 80 registers.  (14 and 16 CTAs per SM -- 72 / 64 registers, the shorter layout of
// the coverage-sample launch makes room for them -- were measured at -1 % / 0 %: the passes are bound by the FMA and ALU
// pipes, not by latency; profiles/r2_notes.md)
constexpr int FB_MIN_CTAS = 12;
template <class PN, int GT, int CPH, bool RENDER, bool REC>
__global__ void __launch_bounds__(FBT, FB_MIN_CTAS) shade_fwd_fallback_kernel(const FwdArgs a, const PN noise_r, const PN noise_a) {
    extern __shared__ __align__(16) unsigned char smem_all[];
    // FBT/32 independent warps per CTA; the coverage-sample launch carries the front of the layout only
    unsigned char* smem_raw = smem_all + (threadIdx.x >> 5) * (CPH == (int)PERT_PH_RAST ? a.L.warp_smem_rast : a.L.warp_smem);
    const int n = 2 * a.worklist[0];
    PN nr = noise_r;
    PN na = noise_a;
    if (a.pb.seed_device) {
        nr.mix(__ldg(a.pb.seed_device));
        na.mix(__ldg(a.pb.seed_device + 1));
    }
#pragma unroll 1
    for (;;) {  // persistent warps fetch half-tiles dynamically
        int i = 0;
        // the aggregation launch walks the list with its own counter
        if ((threadIdx.x & 31) == 0) i = n > 0 ? atomicAdd(a.worklist + ((CPH & PERT_PH_RAST) ? 1 : 2), 1) : 0;
        i = __shfl_sync(FULL, i, 0);
        if (i >= n) break;
        const int64_t tile = (int64_t)a.worklist[4 + (i >> 1)] * 2 + (i & 1);
        if (tile < a.L.ntiles)
            shade_fwd_tile<PN, PN, GT, false, false, CPH, 0, false, RENDER, REC>(a, nr, na, tile, smem_raw, threadIdx.x & 31);
        __syncwarp();
    }
}

template <class NR, class NA, int GT, bool PHASED, bool DEFER, int SCORE, bool WOVR, bool RENDER>
static int launch_t(const FwdArgs& a, const NR& nr, const NA& na, cudaStream_t st) {
    const size_t smem = (size_t)a.L.warp_smem;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(shade_fwd_kernel<NR, NA, GT, PHASED, DEFER, SCORE, WOVR, RENDER>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    shade_fwd_kernel<NR, NA, GT, PHASED, DEFER, SCORE, WOVR, RENDER><<<(unsigned)a.L.ntiles, FNT, smem, st>>>(a, nr, na);
    return (int)cudaGetLastError();
}

template <class PN, int GT, int CPH, bool RENDER, bool REC = false>
static int launch_fallback_ph(const FwdArgs& a, const PN& nr, const PN& na, cudaStream_t st) {
    const size_t smem = (size_t)(CPH == (int)PERT_PH_RAST ? a.L.warp_smem_rast : a.L.warp_smem) * (FBT / 32);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(shade_fwd_fallback_kernel<PN, GT, CPH, RENDER, REC>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    shade_fwd_fallback_kernel<PN, GT, CPH, RENDER, REC>
        <<<resident_grid(shade_fwd_fallback_kernel<PN, GT, CPH, RENDER, REC>, FBT, smem), FBT, smem, st>>>(a, nr, na);
    return (int)cudaGetLastError();
}

// with a tile blob (training) the aggregation launch takes the valid lists from the fallback records
template <class PN, int GT, bool RENDER>
static int launch_fallback(const FwdArgs& a, const PN& nr, const PN& na, cudaStream_t st) {
    const int rc = launch_fallback_ph<PN, GT, PERT_PH_RAST, RENDER>(a, nr, na, st);
    if (rc) return rc;
    if constexpr (!RENDER) {
        if (a.blob) return launch_fallback_ph<PN, GT, PERT_PH_AGG | PERT_PH_BLEND, false, true>(a, nr, na, st);
    }
    return launch_fallback_ph<PN, GT, PERT_PH_AGG | PERT_PH_BLEND, RENDER>(a, nr, na, st);
}

// all phases in one launch, lanes per pixel known at compile time
template <class PN, bool DEFER, bool RENDER>
static int launch_main(const FwdArgs& a, const PN& pr, const PN& pa, cudaStream_t st) {
    switch (a.L.G) {
        case 1: return launch_t<PN, PN, 1, false, DEFER, 0, false, RENDER>(a, pr, pa, st);
        case 2: return launch_t<PN, PN, 2, false, DEFER, 0, false, RENDER>(a, pr, pa, st);
        case 4: return launch_t<PN, PN, 4, false, DEFER, 0, false, RENDER>(a, pr, pa, st);
        default: return launch_t<PN, PN, 8, false, DEFER, 0, false, RENDER>(a, pr, pa, st);
    }
}

// production path (in-kernel Gaussian noise in both stages, all phases in one launch); PN = the Philox variant
template <class PN, bool RENDER>
static int launch_production(const FwdArgs& a, const FwdArgs* fb, cudaStream_t st) {
    const PN pr(a.pb.seed_rast, 0, a.pb.pixel_offset), pa(a.pb.seed_agg, 1, a.pb.pixel_offset);
    if (!fb) return launch_main<PN, false, RENDER>(a, pr, pa, st);
    // sparse-first main pass: defers the tiles the compound sampler is worth running on
    const int rc = launch_main<PN, true, RENDER>(a, pr, pa, st);
    if (rc) return rc;
    switch (fb->L.G) {  // sparse-first mode: half-size tiles for whatever did not fit
        case 2: return launch_fallback<PN, 2, RENDER>(*fb, pr, pa, st);
        case 4: return launch_fallback<PN, 4, RENDER>(*fb, pr, pa, st);
        case 8: return launch_fallback<PN, 8, RENDER>(*fb, pr, pa, st);
        default: return launch_fallback<PN, 16, RENDER>(*fb, pr, pa, st);
    }
}

// One estimator pair: the Gaussian pair (PN = PhiloxNoise), the Cauchy pair (PERT_F_CAUCHY: PN = PhiloxCauchy, SCORE = 1)
// or the pair without control variates (PERT_F_NO_VR: PN = PhiloxNoise, WOVR).  Explicit noise in either stage (PN = the
// in-kernel stream of the other), the Cauchy pair and the pair without control variates run the dense instantiation with
// runtime lanes per pixel; in training it carries the phase-split code, for single and phase-split calls alike.  Unbounded
// Cauchy noise turns off every skip of the Gaussian path (kBounded): each valid entry draws all its coverage samples and
// every finite logit takes part in the argmax.  The pair without control variates keeps the two skips that stay exact for
// it, entries with x < -sigma*Umax and logits that cannot win.  In-kernel Gaussian noise runs the production kernels, or in
// training the phase-split ones of the sample-sharded job.  PHASED: the instantiations carry the phase-split code; always in
// training, in the render only for the phase calls of pert_shade_render_phase.
template <class PN, int SCORE, bool WOVR, bool RENDER, bool PHASED = !RENDER>
static int launch_pair(const FwdArgs& a, const FwdArgs* fb, cudaStream_t st) {
    const bool er = a.pb.noise_rast != nullptr, ea = a.pb.noise_agg != nullptr;
    PN pr(a.pb.seed_rast, 0, a.pb.pixel_offset), pa(a.pb.seed_agg, 1, a.pb.pixel_offset);
    ExplicitNoise xr{a.pb.noise_rast, a.L.P, a.pb.K, a.pb.S_rast}, xa{a.pb.noise_agg, a.L.P, a.pb.K + 1, a.pb.S_agg};
    if (er && ea) return launch_t<ExplicitNoise, ExplicitNoise, 0, PHASED, false, SCORE, WOVR, RENDER>(a, xr, xa, st);
    if (er) return launch_t<ExplicitNoise, PN, 0, PHASED, false, SCORE, WOVR, RENDER>(a, xr, pa, st);
    if (ea) return launch_t<PN, ExplicitNoise, 0, PHASED, false, SCORE, WOVR, RENDER>(a, pr, xa, st);
    if constexpr (SCORE || WOVR) {
        return launch_t<PN, PN, 0, PHASED, false, SCORE, WOVR, RENDER>(a, pr, pa, st);
    } else {
        if constexpr (PHASED) {
            const uint32_t all = PERT_PH_RAST | PERT_PH_AGG | PERT_PH_BLEND;
            if ((a.pb.flags & all) != all || a.hist != nullptr) {  // compile-time lanes per pixel for the benchmark geometries
                switch (a.L.G) {
                    case 4: return launch_t<PN, PN, 4, true, false, 0, false, RENDER>(a, pr, pa, st);
                    case 8: return launch_t<PN, PN, 8, true, false, 0, false, RENDER>(a, pr, pa, st);
                    default: return launch_t<PN, PN, 0, true, false, 0, false, RENDER>(a, pr, pa, st);
                }
            }
        }
        return (a.pb.flags & PERT_F_PHILOX7) ? launch_production<PhiloxNoise7, RENDER>(a, fb, st)
                                             : launch_production<PhiloxNoise, RENDER>(a, fb, st);
    }
}

int launch_shade_fwd(const FwdArgs& a, const FwdArgs* fb, cudaStream_t st) {
    if (a.pb.flags & PERT_F_CAUCHY) return launch_pair<PhiloxCauchy, 1, false, false>(a, fb, st);
    if (a.pb.flags & PERT_F_NO_VR) return launch_pair<PhiloxNoise, 0, true, false>(a, fb, st);
    return launch_pair<PhiloxNoise, 0, false, false>(a, fb, st);
}

// The forward with RENDER = true (shade_fwd_tile): nothing saved for backward.  A single call runs the single-call
// instantiations; a call with a phase bit (pert_shade_render_phase: exactly one) the phase-split ones.  The pair without
// control variates renders on the Gaussian per-sample path (cabi.cu), whose counts, histogram and image it shares.
int launch_shade_render(const FwdArgs& a, const FwdArgs* fb, cudaStream_t st) {
    const bool phased = (a.pb.flags & (PERT_PH_RAST | PERT_PH_AGG | PERT_PH_BLEND)) != 0;
    if (a.pb.flags & PERT_F_CAUCHY)
        return phased ? launch_pair<PhiloxCauchy, 1, false, true, true>(a, fb, st) : launch_pair<PhiloxCauchy, 1, false, true>(a, fb, st);
    return phased ? launch_pair<PhiloxNoise, 0, false, true, true>(a, fb, st) : launch_pair<PhiloxNoise, 0, false, true>(a, fb, st);
}

}  // namespace pert
