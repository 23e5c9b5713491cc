// C ABI of libpertshade.so (include/pertshade.h): argument validation and launch geometry.  Nothing
// here allocates, frees, retains or synchronises; every launch goes to the caller's stream.
#include <math.h>

#include "kernels.h"

using namespace pert;

static thread_local const char* g_last_cuda = "none";

static int cuda_fail(int e) {
    g_last_cuda = cudaGetErrorName((cudaError_t)e);
    return PERT_E_CUDA;
}
static int cuda_rc(int e) { return e == 0 ? PERT_OK : cuda_fail(e); }

extern "C" int pert_version(void) { return PERT_ABI_VERSION; }

extern "C" uint32_t pert_shade_fused_flags(void) {
    return PERT_F_NO_SKIP | PERT_F_SKIP_DEAD_NOISE | PERT_F_PER_SAMPLE_NOISE | PERT_F_CAUCHY | PERT_F_NO_VR | PERT_F_PHILOX7;
}

extern "C" const char* pert_last_cuda_error(void) { return g_last_cuda; }

extern "C" const char* pert_strerror(int code) {
    switch (code) {
        case PERT_OK: return "ok";
        case PERT_E_NULL: return "required pointer is NULL";
        case PERT_E_SHAPE: return "bad shape";
        case PERT_E_UNSUPPORTED: return "K or S not supported by the kernels";
        case PERT_E_ALIGN: return "pointer not aligned";
        case PERT_E_SAMPLES: return "bad sample shard (begin must be a multiple of 4, begin < end <= S)";
        case PERT_E_CUDA: return "CUDA error";
        case PERT_E_SCALAR: return "sigma, gamma and alpha must be finite and > 0";
        default: return "unknown error";
    }
}

// pixels per warp tile: a power of two in [4, 32] with about 512 fragment entries per tile
static int pick_tp(int K) {
    if (K <= 16) return 32;
    if (K <= 32) return 16;
    if (K <= 64) return 8;
    return 4;
}

// Smallest t = |x|/sigma handled by the compound coverage sampler for n local samples: flip probability
// p = Phi(-t) <= min(0.2 [beyond that the per-sample loop is as cheap], 1 - exp(-80/n) [(1-p)^n must not
// underflow], 48/n [serial flips per lane]).
static double tail_quantile(double p) {  // t with Phi(-t) = p, 0 < p <= 0.5
    double lo = 0.0, hi = 8.0;
    for (int i = 0; i < 60; ++i) {
        const double mid = 0.5 * (lo + hi);
        if (0.5 * erfc(mid * 0.7071067811865476) > p) lo = mid; else hi = mid;
    }
    return hi;
}
static float compound_threshold(int n) {
    double pmax = 0.2;
    if (n > 0) {
        pmax = fmin(pmax, 1.0 - exp(-80.0 / n));
        pmax = fmin(pmax, 48.0 / n);
    }
    return (float)tail_quantile(pmax);
}
// bucket edges of the compound sampler: expected flips n p = 3 and 0.25
static void compound_buckets(int n, float t_compound, float* out) {
    const double f0 = 3.0, f1 = 0.25;
    for (int i = 0; i < 2; ++i) {
        const double p = (i == 0 ? f0 : f1) / (n > 0 ? n : 1);
        float t = p >= 0.5 ? 0.0f : (float)tail_quantile(p);
        if (t < t_compound) t = t_compound;
        out[i] = t;
    }
    if (out[1] < out[0]) out[1] = out[0];
}

static int check_problem(const pert_problem* pb) {
    if (!pb) return PERT_E_NULL;
    if (pb->N <= 0 || pb->H <= 0 || pb->W <= 0 || pb->K <= 0) return PERT_E_SHAPE;
    if (pb->K > 1023) return PERT_E_UNSUPPORTED;
    if (pb->N * pb->H * pb->W >= ((int64_t)1 << 31) / (pb->K + 1)) return PERT_E_UNSUPPORTED;  // 32-bit pixel·logit indices per call
    if (pb->S_rast <= 0 || pb->S_agg <= 0 || pb->S_rast > 65535 || pb->S_agg > (1 << 24)) return PERT_E_UNSUPPORTED;
    if (pb->depth_len != 1 && pb->depth_len != pb->N) return PERT_E_SHAPE;
    if (!(pb->sigma > 0.f) || !(pb->gamma > 0.f) || !(pb->alpha > 0.f) || isinf(pb->sigma) || isinf(pb->gamma) ||
        isinf(pb->alpha))
        return PERT_E_SCALAR;
    if ((pb->s_rast_begin & 3) || pb->s_rast_begin < 0 || pb->s_rast_begin >= pb->s_rast_end || pb->s_rast_end > pb->S_rast)
        return PERT_E_SAMPLES;
    if ((pb->s_agg_begin & 3) || pb->s_agg_begin < 0 || pb->s_agg_begin >= pb->s_agg_end || pb->s_agg_end > pb->S_agg)
        return PERT_E_SAMPLES;
    if (!pb->pix_to_face || !pb->zbuf || !pb->dists || !pb->znear || !pb->zfar) return PERT_E_NULL;
    if (pb->face_colors && (pb->num_faces <= 0 || pb->num_faces > 0x7fffffff / 3)) return PERT_E_SHAPE;
    if ((uintptr_t)pb->face_colors & 3) return PERT_E_ALIGN;
    if ((uintptr_t)pb->seed_device & 7) return PERT_E_ALIGN;
    if (((uintptr_t)pb->pix_to_face & 7) || ((uintptr_t)pb->zbuf & 3) || ((uintptr_t)pb->dists & 3)) return PERT_E_ALIGN;
    return PERT_OK;
}

static Launch make_launch(const pert_problem* pb, int tp) {
    Launch L;
    L.tp = tp;
    L.G = 32 / L.tp;
    L.gshift = 0;
    while ((1 << L.gshift) < L.G) L.gshift++;
    L.P = pb->N * pb->H * pb->W;
    L.HW = pb->H * pb->W;
    L.ntiles = (L.P + L.tp - 1) / L.tp;
    L.win_bytes = pert_winner_bytes(pb->K);
    L.sa_loc = pb->s_agg_end - pb->s_agg_begin;
    int sc = 1024 / L.tp;  // c_s staging: about 4 KB per warp
    const int s32 = (L.sa_loc + 31) & ~31;
    if (sc > s32) sc = s32;
    L.sc = sc;
    L.nchunks = (L.sa_loc + sc - 1) / sc;
    const int nq_r = ((pb->s_rast_end + 3) >> 2) - (pb->s_rast_begin >> 2), nq_a = (L.sa_loc + 3) >> 2;
    auto lg2 = [](int v) { int s = 0; while ((1 << s) < v) s++; return s; };
    L.lpe_r = pow2_ceil(nq_r) < 32 ? pow2_ceil(nq_r) : 32;
    L.lpe_r_shift = lg2(L.lpe_r);
    L.lpe_a = pow2_ceil(nq_a) < 32 ? pow2_ceil(nq_a) : 32;
    L.lpe_a_shift = lg2(L.lpe_a);
    L.lpp = pow2_floor(nq_a) < 32 ? pow2_floor(nq_a) : 32;
    L.lpp_shift = lg2(L.lpp);
    L.cap = L.tp * pb->K;
    L.warp_smem = 0;
    L.warp_smem_rast = 0;
    // 128-bit accesses on the tile rows need every tile to start on a 16-byte boundary in the fp32 tensors
    L.vec_ok = ((L.tp * pb->K) & 3) == 0;
    L.invK = 1.0f / (float)pb->K;
    L.gal = pb->gamma / pb->alpha;
    L.inv_sigma = 1.0f / pb->sigma;
    L.invSg = 1.0f / ((float)pb->S_agg * pb->gamma);
    L.inv_sr = 1.0f / ((float)pb->S_rast * pb->sigma);
    L.invS = 1.0f / (float)pb->S_agg;
    L.inv_gamma = 1.0f / pb->gamma;
    L.t_compound = compound_threshold(pb->s_rast_end - pb->s_rast_begin);
    compound_buckets(pb->s_rast_end - pb->s_rast_begin, L.t_compound, L.t_bucket);
    L.lean = false;
    return L;
}

// Sparse-first mode (production default when the caller passes a work list): the main pass sizes its
// compact arrays for HALF the entries of a tile -- real fragments fill a few percent -- which halves the
// shared memory per warp; a tile with more valid entries is put on the work list and redone by the
// fallback pass as two half-size tiles.
// Sparse-first geometry: the main pass takes tiles of TWICE the pixels (fewer per-tile fixed costs, better
// lane packing in the sampling loops: -10 % instructions) with compact arrays for 40 % of the entries of a
// normal tile; the fallback pass redoes an overflowing tile as two normal tiles with full capacity.
static int sparse_tp(int K, int64_t P) {
    int tp = 2 * pick_tp(K);
    if (tp > 32) tp = 32;
    // small jobs: prefer enough tiles to fill the GPU (SMs x ~24 resident warps) over double-size tiles
    if (tp > pick_tp(K) && (P + tp - 1) / tp < (int64_t)sm_count() * 24) tp = pick_tp(K);
    // ... and jobs of few pixels with many samples (BASELINE config 4: 128^2 pixels, S = 4096) want every SM busy: halve
    // the tile while there are fewer than ~16 warps per SM (6.6 -> 3.6 ms at config 4)
    while (tp > 4 && (P + tp - 1) / tp < (int64_t)sm_count() * 16) tp >>= 1;
    return tp;
}
// tile of the launches that do not run sparse-first (phase-split / explicit-noise / per-sample jobs): the same rule for
// jobs of few pixels (a sample shard of BASELINE config 4 is 128^2 pixels x 512 samples)
static int dense_tp(int K, int64_t P) {
    int tp = pick_tp(K);
    while (tp > 4 && (P + tp - 1) / tp < (int64_t)sm_count() * 16) tp >>= 1;
    return tp;
}
static int sparse_cap(int K, int tp) {
    int cap = tp * K / 5;
    cap = (cap + 7) & ~7;  // u16 arrays are copied as 32-bit words
    if (cap < 32) cap = 32;
    if (cap > tp * K) cap = (tp * K + 1) & ~1;
    return cap;
}

static bool sparse_first_ok(const pert_problem* pb, const void* worklist, bool all_phases) {
    if (!worklist || !all_phases || pb->noise_rast || pb->noise_agg) return false;
    if (pb->flags & (PERT_F_NO_SKIP | PERT_F_PER_SAMPLE_NOISE | PERT_F_CAUCHY | PERT_F_NO_VR)) return false;  // need logits dense in j
    return true;
}

// flags the fused entry points cannot combine with PERT_F_CAUCHY: another Gaussian stream, the ablation without control
// variates, the expectation shortcut for never-winning logits (a Gaussian identity) and the forward-only noises
static bool cauchy_flags_bad(uint32_t f) {
    return (f & PERT_F_CAUCHY) &&
           (f & (PERT_F_PHILOX7 | PERT_F_NO_VR | PERT_F_SKIP_DEAD_NOISE | PERT_F_UNIFORM | PERT_F_GUMBEL));
}

// flags the fused entry points cannot combine with PERT_F_NO_VR: its kernels draw the Philox4x32-10 stream of every
// sample (the shortcut for never-winning logits is a variance-reduced estimator's), and the forward-only noises
static bool no_vr_flags_bad(uint32_t f) {
    return (f & PERT_F_NO_VR) && (f & (PERT_F_PHILOX7 | PERT_F_SKIP_DEAD_NOISE | PERT_F_UNIFORM | PERT_F_GUMBEL));
}

extern "C" int64_t pert_num_tiles(const pert_problem* pb) {
    if (!pb || pb->K <= 0) return 0;
    const int64_t P = pb->N * pb->H * pb->W;
    const int a = dense_tp(pb->K, P), b = sparse_tp(pb->K, P);
    const int tp = a < b ? a : b;  // the finest tile geometry any launch of this problem uses
    return (P + tp - 1) / tp;
}

extern "C" int pert_winner_bytes(int32_t K) { return (K + 1 <= 256) ? 1 : 2; }

// The tile_blob buffer: one tile blob per tile of the sparse-first main pass, then one fallback record per half-tile, for
// every tile (each one may be deferred).  Offset of the records region in 32-bit words:
static int64_t blob_records_off(int K, int64_t P) {
    const int tp = sparse_tp(K, P);
    return ((P + tp - 1) / tp) * (int64_t)blob_words(tp, sparse_cap(K, tp));
}

extern "C" int64_t pert_blob_bytes(const pert_problem* pb) {
    if (!pb || pb->K <= 0) return 0;
    const int64_t P = pb->N * pb->H * pb->W;
    const int tp = sparse_tp(pb->K, P);
    const int64_t records = 2 * ((P + tp - 1) / tp) * (int64_t)fbrec_words(tp / 2, tp / 2 * pb->K);
    return (blob_records_off(pb->K, P) + records) * 4;
}

static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

// Launch records of a single forward call: `a` (pointers set) gets the main pass's tile geometry and, in sparse-first mode,
// `fb` the fallback pass's (half-size tiles, full capacity).  Returns 1 in sparse-first mode, 0 without it, or a PERT_E_*.
static int fwd_launch_records(FwdArgs& a, FwdArgs& fb, bool sparse) {
    const int64_t P = a.pb.N * a.pb.H * a.pb.W;
    if (sparse) {  // the fallback pass runs FBT/32 warps per CTA: its tiles must fit that many times
        SmemLayout t;
        const int tp2 = sparse_tp(a.pb.K, P) / 2;
        fwd_smem_layout(tp2, tp2 * a.pb.K, t);
        if ((size_t)t.bytes * (FBT / 32) > 200 * 1024) sparse = false;
    }
    a.L = make_launch(&a.pb, sparse ? sparse_tp(a.pb.K, P) : dense_tp(a.pb.K, P));
    a.L.vec_ok = a.L.vec_ok && aligned16(a.pb.pix_to_face);
    if (sparse) a.L.cap = sparse_cap(a.pb.K, a.L.tp);
    fwd_smem_layout(a.L.tp, a.L.cap, a.L.sm);
    a.L.warp_smem = a.L.sm.bytes;
    if ((size_t)a.L.warp_smem > 200 * 1024) return PERT_E_UNSUPPORTED;
    if (a.L.ntiles > 0x7fffffff) return PERT_E_UNSUPPORTED;
    if (!sparse) return 0;
    fb = a;
    fb.blob = a.blob ? a.blob + blob_records_off(a.pb.K, P) : nullptr;
    fb.L = make_launch(&a.pb, a.L.tp / 2);
    fb.L.vec_ok = fb.L.vec_ok && aligned16(a.pb.pix_to_face);
    fb.L.warp_smem_rast = fwd_smem_layout(fb.L.tp, fb.L.cap, fb.L.sm);
    fb.L.warp_smem = fb.L.sm.bytes;
    return 1;
}

extern "C" int pert_shade_fwd(const pert_problem* pb_in, float* image, uint16_t* counts, float* rsum, void* winners,
                              uint16_t* pixstate, int32_t* hist, int32_t* worklist, void* tile_blob, void* stream) {
    int rc = check_problem(pb_in);
    if (rc) return rc;
    FwdArgs a;
    a.pb = *pb_in;
    if (!(a.pb.flags & (PERT_PH_RAST | PERT_PH_AGG | PERT_PH_BLEND))) a.pb.flags |= PERT_PH_RAST | PERT_PH_AGG | PERT_PH_BLEND;
    const uint32_t f = a.pb.flags;
    if (!counts) return PERT_E_NULL;
    if ((f & PERT_PH_RAST) && !rsum) return PERT_E_NULL;
    if ((f & PERT_PH_AGG) && (!winners || !pixstate)) return PERT_E_NULL;
    if ((f & PERT_PH_BLEND) && (!image || (!a.pb.colors && !a.pb.face_colors))) return PERT_E_NULL;
    if (((f & PERT_PH_AGG) != 0) != ((f & PERT_PH_BLEND) != 0) && !hist) return PERT_E_NULL;
    if (((uintptr_t)image & 15) || ((uintptr_t)counts & 1) || ((uintptr_t)rsum & 3) || ((uintptr_t)hist & 3) ||
        ((uintptr_t)a.pb.colors & 3) || ((uintptr_t)pixstate & 1) || ((uintptr_t)winners & 3))
        return PERT_E_ALIGN;
    if ((uintptr_t)worklist & 15) return PERT_E_ALIGN;
    const uint32_t all = PERT_PH_RAST | PERT_PH_AGG | PERT_PH_BLEND;
    if ((f & PERT_F_PHILOX7) && ((f & all) != all || hist || a.pb.noise_rast || a.pb.noise_agg)) return PERT_E_UNSUPPORTED;
    if (cauchy_flags_bad(f) || no_vr_flags_bad(f)) return PERT_E_UNSUPPORTED;
    a.image = image;
    a.counts = counts;
    a.rsum = rsum;
    a.winners = winners;
    a.pixstate = pixstate;
    a.hist = hist;
    a.worklist = worklist;
    a.blob = (int32_t*)tile_blob;  // the fallback pass's records follow the tile blobs (fwd_launch_records)
    FwdArgs fb;
    rc = fwd_launch_records(a, fb, sparse_first_ok(&a.pb, worklist, (f & all) == all && !hist));
    if (rc < 0) return rc;
    const bool sparse = rc == 1;
    if ((uintptr_t)tile_blob & 15) return PERT_E_ALIGN;
    if (!sparse) a.blob = nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    if (!sparse) return cuda_rc(launch_shade_fwd(a, nullptr, st));
    cudaError_t e = cudaMemsetAsync(worklist, 0, 16, st);
    if (e != cudaSuccess) return cuda_fail((int)e);
    return cuda_rc(launch_shade_fwd(a, &fb, st));
}

extern "C" int pert_shade_render(const pert_problem* pb_in, float* image, uint16_t* counts_ws, int32_t* worklist,
                                 void* stream) {
    int rc = check_problem(pb_in);
    if (rc) return rc;
    FwdArgs a = {};
    a.pb = *pb_in;
    const uint32_t f = a.pb.flags;
    // one call renders every sample: the phase-split (sample-sharded) forward has no forward-only form
    if (f & (PERT_PH_RAST | PERT_PH_AGG | PERT_PH_BLEND | PERT_PH_BWD_SAMPLE | PERT_PH_BWD_FINISH)) return PERT_E_UNSUPPORTED;
    if (a.pb.s_rast_begin != 0 || a.pb.s_rast_end != a.pb.S_rast || a.pb.s_agg_begin != 0 || a.pb.s_agg_end != a.pb.S_agg)
        return PERT_E_UNSUPPORTED;
    if (!image || (!a.pb.colors && !a.pb.face_colors)) return PERT_E_NULL;
    if (((uintptr_t)image & 15) || ((uintptr_t)counts_ws & 1) || ((uintptr_t)a.pb.colors & 3) || ((uintptr_t)worklist & 15))
        return PERT_E_ALIGN;
    if ((f & PERT_F_PHILOX7) && (a.pb.noise_rast || a.pb.noise_agg)) return PERT_E_UNSUPPORTED;
    if (cauchy_flags_bad(f) || no_vr_flags_bad(f)) return PERT_E_UNSUPPORTED;
    // the pair without control variates differs from the Gaussian pair in rsum only, which a render does not produce: its
    // counts, histogram and image are those of the Gaussian per-sample path (no compound sampler), on the same tiles
    if (f & PERT_F_NO_VR) a.pb.flags |= PERT_F_PER_SAMPLE_NOISE;
    // the fallback pass of the sparse-first mode keeps its counts in counts_ws; no other mode touches it
    const bool sparse_ok = sparse_first_ok(&a.pb, worklist, true);
    if (sparse_ok && !counts_ws) return PERT_E_NULL;
    a.image = image;
    a.counts = counts_ws;
    a.worklist = worklist;
    FwdArgs fb;
    rc = fwd_launch_records(a, fb, sparse_ok);
    if (rc < 0) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (rc == 0) return cuda_rc(launch_shade_render(a, nullptr, st));
    cudaError_t e = cudaMemsetAsync(worklist, 0, 16, st);
    if (e != cudaSuccess) return cuda_fail((int)e);
    return cuda_rc(launch_shade_render(a, &fb, st));
}

extern "C" int pert_shade_render_phase(const pert_problem* pb_in, float* image, uint16_t* counts, int32_t* hist,
                                       void* stream) {
    int rc = check_problem(pb_in);
    if (rc) return rc;
    FwdArgs a = {};
    a.pb = *pb_in;
    const uint32_t f = a.pb.flags;
    const uint32_t ph = f & (PERT_PH_RAST | PERT_PH_AGG | PERT_PH_BLEND);
    // one forward phase per call (the collectives sit between them); backward phases have no forward-only form
    if (ph == 0 || (ph & (ph - 1)) || (f & (PERT_PH_BWD_SAMPLE | PERT_PH_BWD_FINISH))) return PERT_E_UNSUPPORTED;
    if (!counts) return PERT_E_NULL;
    if (ph != PERT_PH_RAST && !hist) return PERT_E_NULL;
    if (ph == PERT_PH_BLEND && (!image || (!a.pb.colors && !a.pb.face_colors))) return PERT_E_NULL;
    if (((uintptr_t)image & 15) || ((uintptr_t)counts & 1) || ((uintptr_t)hist & 3) || ((uintptr_t)a.pb.colors & 3))
        return PERT_E_ALIGN;
    if (f & PERT_F_PHILOX7) return PERT_E_UNSUPPORTED;
    if (cauchy_flags_bad(f) || no_vr_flags_bad(f)) return PERT_E_UNSUPPORTED;
    if (f & PERT_F_NO_VR) a.pb.flags |= PERT_F_PER_SAMPLE_NOISE;  // as in pert_shade_render
    a.image = image;
    a.counts = counts;
    a.hist = hist;
    FwdArgs fb;
    rc = fwd_launch_records(a, fb, false);  // the tiles of pert_shade_fwd's phase calls
    if (rc < 0) return rc;
    return cuda_rc(launch_shade_render(a, nullptr, (cudaStream_t)stream));
}

extern "C" int pert_shade_bwd(const pert_problem* pb_in, const float* grad_image, const uint16_t* counts,
                              const float* rsum, const void* winners, const uint16_t* pixstate, float* grad_dists,
                              float* grad_zbuf, float* grad_colors, float* scalar_partials, float* grad_scalars,
                              float* acc, float* pixstat, const int32_t* hist, int32_t* worklist,
                              const void* tile_blob, void* stream) {
    int rc = check_problem(pb_in);
    if (rc) return rc;
    BwdArgs a;
    a.pb = *pb_in;
    if (!(a.pb.flags & (PERT_PH_BWD_SAMPLE | PERT_PH_BWD_FINISH))) a.pb.flags |= PERT_PH_BWD_SAMPLE | PERT_PH_BWD_FINISH;
    const uint32_t f = a.pb.flags;
    const bool smp = f & PERT_PH_BWD_SAMPLE, fin = f & PERT_PH_BWD_FINISH;
    if (!grad_image || !counts || !rsum || !pixstate || (!a.pb.colors && !a.pb.face_colors)) return PERT_E_NULL;
    if (smp && !winners) return PERT_E_NULL;
    if (fin && (!grad_dists || !grad_zbuf || !scalar_partials || !grad_scalars)) return PERT_E_NULL;
    if (smp != fin && (!acc || !pixstat)) return PERT_E_NULL;
    if (fin && !smp && grad_colors && !hist) return PERT_E_NULL;
    if (((uintptr_t)grad_image & 15) || ((uintptr_t)grad_colors & 3) || ((uintptr_t)grad_dists & 3) ||
        ((uintptr_t)grad_zbuf & 3) || ((uintptr_t)counts & 1) || ((uintptr_t)rsum & 3) || ((uintptr_t)pixstate & 1) ||
        ((uintptr_t)scalar_partials & 15) || ((uintptr_t)acc & 3) || ((uintptr_t)pixstat & 3) || ((uintptr_t)hist & 3))
        return PERT_E_ALIGN;
    if ((uintptr_t)worklist & 15) return PERT_E_ALIGN;
    if ((f & PERT_F_PHILOX7) && (!(smp && fin) || hist || a.pb.noise_agg)) return PERT_E_UNSUPPORTED;
    if (cauchy_flags_bad(f) || no_vr_flags_bad(f)) return PERT_E_UNSUPPORTED;
    bool sparse = sparse_first_ok(&a.pb, worklist, smp && fin && !hist);
    if (sparse) {  // the fallback pass runs FBT/32 warps per CTA: its tiles must fit that many times
        const int tp2 = sparse_tp(a.pb.K, a.pb.N * a.pb.H * a.pb.W) / 2;
        const Launch t = make_launch(&a.pb, tp2);
        SmemLayout sl;
        bwd_smem_layout(tp2, a.pb.K, t.cap, t.sc, t.nchunks, t.win_bytes, false, true, sl);
        if ((size_t)sl.bytes * (FBT / 32) > 200 * 1024) sparse = false;
    }
    const bool ptr_ok = aligned16(a.pb.pix_to_face) && aligned16(grad_dists) && aligned16(grad_zbuf) &&
                        (a.pb.face_colors || aligned16(grad_colors));
    a.L = make_launch(&a.pb, sparse ? sparse_tp(a.pb.K, a.pb.N * a.pb.H * a.pb.W) : dense_tp(a.pb.K, a.pb.N * a.pb.H * a.pb.W));
    a.L.vec_ok = a.L.vec_ok && ptr_ok;
    if (sparse) a.L.cap = sparse_cap(a.pb.K, a.L.tp);
    if (a.L.win_bytes == 2 && ((uintptr_t)winners & 1)) return PERT_E_ALIGN;
    bwd_smem_layout(a.L.tp, a.pb.K, a.L.cap, a.L.sc, a.L.nchunks, a.L.win_bytes, sparse, a.L.lean, a.L.sm);
    a.L.warp_smem = a.L.sm.bytes;
    if ((size_t)a.L.warp_smem > 200 * 1024) return PERT_E_UNSUPPORTED;
    if (a.L.ntiles > 0x7fffffff) return PERT_E_UNSUPPORTED;
    a.grad_image = grad_image;
    a.counts = counts;
    a.rsum = rsum;
    a.winners = winners;
    a.pixstate = pixstate;
    a.grad_dists = grad_dists;
    a.grad_zbuf = grad_zbuf;
    a.grad_colors = grad_colors;
    a.partials = scalar_partials;
    a.acc = acc;
    a.pixstat = pixstat;
    a.hist = hist;
    a.worklist = worklist;
    if ((uintptr_t)tile_blob & 15) return PERT_E_ALIGN;
    a.blob = sparse ? (const int32_t*)tile_blob : nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    if (!sparse) return cuda_rc(launch_shade_bwd(a, nullptr, grad_scalars, st));
    BwdArgs fb = a;  // fallback pass: half-size tiles, full capacity, dense per-logit arrays
    fb.blob = a.blob ? a.blob + blob_records_off(a.pb.K, a.L.P) : nullptr;
    fb.L = make_launch(&a.pb, a.L.tp / 2);
    fb.L.vec_ok = fb.L.vec_ok && ptr_ok;
    fb.L.lean = true;  // pair list in the counts array; the winners ARE staged (+3 %), the layout still fits 12 CTAs per SM
    bwd_smem_layout(fb.L.tp, a.pb.K, fb.L.cap, fb.L.sc, fb.L.nchunks, fb.L.win_bytes, false, fb.L.lean, fb.L.sm);
    fb.L.warp_smem = fb.L.sm.bytes;
    cudaError_t e = cudaMemsetAsync(worklist, 0, 16, st);
    if (e != cudaSuccess) return cuda_fail((int)e);
    return cuda_rc(launch_shade_bwd(a, &fb, grad_scalars, st));
}

// ---- SoftRas pair (SoftRast + SoftAgg), deterministic -----------------------------------------------
static int soft_launch_record(pert_problem& pb, Launch& L, bool bwd, bool ptr_ok) {
    // sample counts are unused on this path; make the shared validation happy
    pb.S_rast = pb.S_agg = 4;
    pb.s_rast_begin = pb.s_agg_begin = 0;
    pb.s_rast_end = pb.s_agg_end = 4;
    pb.noise_rast = pb.noise_agg = nullptr;
    pb.face_colors = nullptr;
    int rc = check_problem(&pb);
    if (rc) return rc;
    if (!pb.colors) return PERT_E_NULL;
    L = make_launch(&pb, pick_tp(pb.K));
    L.vec_ok = L.vec_ok && ptr_ok;
    soft_smem_layout(L.tp, pb.K, bwd, L.sm);
    L.warp_smem = L.sm.bytes;
    if ((size_t)L.warp_smem > 200 * 1024) return PERT_E_UNSUPPORTED;
    return PERT_OK;
}

extern "C" int pert_soft_shade_fwd(const pert_problem* pb_in, float* image, void* stream) {
    if (!pb_in || !image) return PERT_E_NULL;
    if ((uintptr_t)image & 15) return PERT_E_ALIGN;
    pert_problem pb = *pb_in;
    Launch L;
    if (int rc = soft_launch_record(pb, L, false, aligned16(pb.pix_to_face))) return rc;
    return cuda_rc(launch_soft_fwd(pb, L, image, (cudaStream_t)stream));
}

extern "C" int pert_soft_shade_bwd(const pert_problem* pb_in, const float* grad_image, float* grad_dists, float* grad_zbuf,
                                   float* grad_colors, float* scalar_partials, float* grad_scalars, void* stream) {
    if (!pb_in || !grad_image || !grad_dists || !grad_zbuf || !scalar_partials || !grad_scalars) return PERT_E_NULL;
    if (((uintptr_t)grad_image & 15) || ((uintptr_t)scalar_partials & 15) || ((uintptr_t)grad_dists & 3) ||
        ((uintptr_t)grad_zbuf & 3) || ((uintptr_t)grad_colors & 3))
        return PERT_E_ALIGN;
    pert_problem pb = *pb_in;
    Launch L;
    const bool ptr_ok = aligned16(pb.pix_to_face) && aligned16(grad_dists) && aligned16(grad_zbuf) && aligned16(grad_colors);
    if (int rc = soft_launch_record(pb, L, true, ptr_ok)) return rc;
    return cuda_rc(launch_soft_bwd(pb, L, grad_image, grad_dists, grad_zbuf, grad_colors, scalar_partials, grad_scalars,
                                   (cudaStream_t)stream));
}

extern "C" int pert_rast_fwd(const float* x, int64_t P, int32_t K, int32_t S, int32_t s_begin, int32_t s_end,
                             float sigma, uint64_t seed, int64_t pixel_offset, const float* noise, uint32_t flags,
                             float* prob, float* rsum, void* stream) {
    if (!x || !prob || !rsum) return PERT_E_NULL;
    if (P <= 0 || K <= 0) return PERT_E_SHAPE;
    if (S <= 0 || S > 65535) return PERT_E_UNSUPPORTED;
    if ((s_begin & 3) || s_begin < 0 || s_begin >= s_end || s_end > S) return PERT_E_SAMPLES;
    if (!(sigma > 0.f) || isinf(sigma)) return PERT_E_SCALAR;
    if ((P * K + 1023) / 1024 > 0x7fffffff) return PERT_E_UNSUPPORTED;
    return cuda_rc(launch_rast_fwd(x, P, K, S, s_begin, s_end, sigma, seed, pixel_offset, noise, flags, prob, rsum,
                                   (cudaStream_t)stream));
}

extern "C" int pert_rast_bwd(const float* grad_l, const float* rsum, int64_t n, int32_t S, float sigma, float* grad_x,
                             float* scalar_partials, float* grad_sigma, void* stream) {
    if (!grad_l || !rsum || !grad_x || !scalar_partials || !grad_sigma) return PERT_E_NULL;
    if (n <= 0 || S <= 0) return PERT_E_SHAPE;
    if (!(sigma > 0.f)) return PERT_E_SCALAR;
    if ((n + 255) / 256 > 0x7fffffff) return PERT_E_UNSUPPORTED;
    return cuda_rc(launch_rast_bwd(grad_l, rsum, n, S, sigma, grad_x, scalar_partials, grad_sigma, (cudaStream_t)stream));
}

extern "C" int pert_argmax_fwd(const float* z, int64_t P, int32_t K1, int32_t S, int32_t s_begin, int32_t s_end,
                               float gamma, uint64_t seed, int64_t pixel_offset, const float* noise, uint32_t flags,
                               float* weights, void* winners, void* stream) {
    if (!z || !weights || !winners) return PERT_E_NULL;
    if (P <= 0 || K1 <= 0) return PERT_E_SHAPE;
    if (K1 > 1024 || S <= 0 || S > (1 << 24)) return PERT_E_UNSUPPORTED;
    if ((s_begin & 3) || s_begin < 0 || s_begin >= s_end || s_end > S) return PERT_E_SAMPLES;
    if (!(gamma > 0.f) || isinf(gamma)) return PERT_E_SCALAR;
    if ((P + NW - 1) / NW > 0x7fffffff) return PERT_E_UNSUPPORTED;
    return cuda_rc(launch_argmax_fwd(z, P, K1, S, s_begin, s_end, gamma, seed, pixel_offset, noise, flags, weights,
                                     winners, (cudaStream_t)stream));
}

extern "C" int pert_argmax_bwd(const float* grad_l, const float* z, const void* winners, int64_t P, int32_t K1,
                               int32_t S, int32_t s_begin, int32_t s_end, float gamma, uint64_t seed,
                               int64_t pixel_offset, const float* noise, uint32_t flags, float* grad_z,
                               float* scalar_partials, float* grad_gamma, void* stream) {
    if (flags & (PERT_F_UNIFORM | PERT_F_GUMBEL)) return PERT_E_UNSUPPORTED;  // forward-only noises (no backward in the reference)
    if (!grad_l || !z || !winners || !grad_z || !scalar_partials || !grad_gamma) return PERT_E_NULL;
    if (P <= 0 || K1 <= 0) return PERT_E_SHAPE;
    if (K1 > 1024 || S <= 0) return PERT_E_UNSUPPORTED;
    if ((s_begin & 3) || s_begin < 0 || s_begin >= s_end || s_end > S) return PERT_E_SAMPLES;
    if (!(gamma > 0.f) || isinf(gamma)) return PERT_E_SCALAR;
    if ((P + NW - 1) / NW > 0x7fffffff) return PERT_E_UNSUPPORTED;
    return cuda_rc(launch_argmax_bwd(grad_l, z, winners, P, K1, S, s_begin, s_end, gamma, seed, pixel_offset, noise,
                                     flags, grad_z, scalar_partials, grad_gamma, (cudaStream_t)stream));
}

extern "C" int pert_seed_advance(uint64_t* seed_device, void* stream) {
    if (!seed_device) return PERT_E_NULL;
    if ((uintptr_t)seed_device & 7) return PERT_E_ALIGN;
    return cuda_rc(launch_seed_advance(seed_device, (cudaStream_t)stream));
}

extern "C" int pert_noise_fill(uint64_t seed, int32_t stage, int64_t P, int32_t slots, int32_t s_begin, int32_t s_end,
                               int64_t pixel_offset, float* out, void* stream) {
    if (!out) return PERT_E_NULL;
    if (P <= 0 || slots <= 0) return PERT_E_SHAPE;
    if ((s_begin & 3) || s_begin < 0 || s_begin >= s_end) return PERT_E_SAMPLES;
    const int qn = ((s_end + 3) >> 2) - (s_begin >> 2);
    if (((int64_t)qn * P * slots + 255) / 256 > 0x7fffffff) return PERT_E_UNSUPPORTED;
    return cuda_rc(launch_noise_fill(seed, stage, P, slots, s_begin, s_end, pixel_offset, out, (cudaStream_t)stream));
}

// atlas: the call brings its own texel source (pert_phong_atlas_*), and none of ph's may be set
static int check_phong(const pert_phong* ph, bool atlas = false) {
    if (!ph) return PERT_E_NULL;
    if (ph->P <= 0 || ph->HW <= 0 || ph->K <= 0 || ph->num_faces <= 0 || ph->P % ph->HW != 0) return PERT_E_SHAPE;
    if (ph->num_faces > 0x7fffffff / 27 || ph->P >= ((int64_t)1 << 32) / ph->K) return PERT_E_UNSUPPORTED;  // 32-bit entry indices
    const bool unlit = ph->flags & PERT_PHONG_UNLIT;
    if (!unlit && ph->light_rows != 1 && ph->light_rows != ph->P / ph->HW) return PERT_E_SHAPE;
    if (!ph->pix_to_face || !ph->bary) return PERT_E_NULL;
    if (!unlit && (!ph->face_verts || !ph->face_normals || !ph->lighting)) return PERT_E_NULL;
    const int sources = (ph->texels != nullptr) + (ph->face_colors != nullptr) + (ph->face_vert_colors != nullptr) + (ph->uv_map != nullptr);
    if (atlas && sources != 0) return PERT_E_UNSUPPORTED;
    if (!atlas && sources != 1) return PERT_E_NULL;
    if (ph->uv_map && (!ph->face_uvs || ph->map_h <= 0 || ph->map_w <= 0 || (ph->map_count != 1 && ph->map_count != ph->P / ph->HW)))
        return PERT_E_SHAPE;
    if (((uintptr_t)ph->uv_map & 3) || ((uintptr_t)ph->face_uvs & 3)) return PERT_E_ALIGN;
    if (((uintptr_t)ph->pix_to_face & 7) || ((uintptr_t)ph->bary & 3) || ((uintptr_t)ph->face_verts & 3) ||
        ((uintptr_t)ph->face_normals & 3) || ((uintptr_t)ph->texels & 3) || ((uintptr_t)ph->face_colors & 3) ||
        ((uintptr_t)ph->lighting & 3) || ((uintptr_t)ph->face_vert_colors & 3))
        return PERT_E_ALIGN;
    return PERT_OK;
}

extern "C" int pert_phong_fwd(const pert_phong* ph, float* colors, void* stream) {
    if (int rc = check_phong(ph)) return rc;
    if (!colors) return PERT_E_NULL;
    if ((uintptr_t)colors & 3) return PERT_E_ALIGN;
    return cuda_rc(launch_phong_fwd(*ph, colors, (cudaStream_t)stream));
}

extern "C" int pert_phong_bwd(const pert_phong* ph, const float* grad_colors, float* grad_texels, float* grad_bary,
                              float* grad_face_verts, float* grad_face_normals, float* grad_lighting, void* stream) {
    if (int rc = check_phong(ph)) return rc;
    if (!grad_colors) return PERT_E_NULL;
    if (((uintptr_t)grad_colors & 3) || ((uintptr_t)grad_texels & 3) || ((uintptr_t)grad_bary & 3) ||
        ((uintptr_t)grad_face_verts & 3) || ((uintptr_t)grad_face_normals & 3) || ((uintptr_t)grad_lighting & 3))
        return PERT_E_ALIGN;
    if (grad_lighting && (ph->flags & PERT_PHONG_UNLIT)) return PERT_E_UNSUPPORTED;
    if (grad_texels || grad_bary || grad_face_verts || grad_face_normals)
        if (int rc = cuda_rc(launch_phong_bwd(*ph, grad_colors, grad_texels, grad_bary, grad_face_verts, grad_face_normals,
                                              (cudaStream_t)stream)))
            return rc;
    if (grad_lighting) return cuda_rc(launch_phong_light_bwd(*ph, grad_colors, grad_lighting, (cudaStream_t)stream));
    return PERT_OK;
}

static int check_phong_atlas(const pert_phong* ph, const float* atlas, int32_t atlas_size) {
    if (int rc = check_phong(ph, true)) return rc;
    if (!atlas) return PERT_E_NULL;
    if (atlas_size <= 0) return PERT_E_SHAPE;
    // 32-bit atlas offsets: num_faces R^2 3 <= 2^31 - 1 (written so that nothing overflows)
    if ((int64_t)atlas_size * atlas_size > 0x7fffffff / 3 / ph->num_faces) return PERT_E_UNSUPPORTED;
    if ((uintptr_t)atlas & 3) return PERT_E_ALIGN;
    return PERT_OK;
}

extern "C" int pert_phong_atlas_fwd(const pert_phong* ph, const float* atlas, int32_t atlas_size, float* colors, void* stream) {
    if (int rc = check_phong_atlas(ph, atlas, atlas_size)) return rc;
    if (!colors) return PERT_E_NULL;
    if ((uintptr_t)colors & 3) return PERT_E_ALIGN;
    return cuda_rc(launch_phong_fwd(*ph, colors, (cudaStream_t)stream, atlas, atlas_size));
}

extern "C" int pert_phong_atlas_bwd(const pert_phong* ph, const float* atlas, int32_t atlas_size, const float* grad_colors,
                                    float* grad_atlas, float* grad_bary, float* grad_face_verts, float* grad_face_normals,
                                    float* grad_lighting, void* stream) {
    if (int rc = check_phong_atlas(ph, atlas, atlas_size)) return rc;
    if (!grad_colors) return PERT_E_NULL;
    if (((uintptr_t)grad_colors & 3) || ((uintptr_t)grad_atlas & 3) || ((uintptr_t)grad_bary & 3) ||
        ((uintptr_t)grad_face_verts & 3) || ((uintptr_t)grad_face_normals & 3) || ((uintptr_t)grad_lighting & 3))
        return PERT_E_ALIGN;
    if (grad_lighting && (ph->flags & PERT_PHONG_UNLIT)) return PERT_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (grad_atlas || grad_bary || grad_face_verts || grad_face_normals)
        if (int rc = cuda_rc(launch_phong_bwd(*ph, grad_colors, grad_atlas, grad_bary, grad_face_verts, grad_face_normals, st, atlas,
                                              atlas_size)))
            return rc;
    if (grad_lighting) return cuda_rc(launch_phong_light_bwd(*ph, grad_colors, grad_lighting, st, atlas, atlas_size));
    return PERT_OK;
}

static int check_raster(const pert_raster* rs) {
    if (!rs) return PERT_E_NULL;
    if (rs->N <= 0 || rs->H <= 0 || rs->W <= 0 || rs->K <= 0 || rs->num_faces <= 0) return PERT_E_SHAPE;
    if (rs->N > 65535 || rs->K > 1023 || rs->num_faces > 0x7fffffff / 9) return PERT_E_UNSUPPORTED;
    if ((int64_t)rs->N * rs->H * rs->W >= ((int64_t)1 << 32) / rs->K) return PERT_E_UNSUPPORTED;
    if (!(rs->blur_radius >= 0.0f) || isinf(rs->blur_radius)) return PERT_E_SCALAR;
    if (!rs->face_verts || !rs->face_start) return PERT_E_NULL;
    if (((uintptr_t)rs->face_verts & 3) || ((uintptr_t)rs->face_start & 7) || ((uintptr_t)rs->face_order & 7)) return PERT_E_ALIGN;
    return PERT_OK;
}

extern "C" int pert_rasterize_fwd(const pert_raster* rs, int64_t* pix_to_face, float* zbuf, float* bary, float* dists,
                                  void* stream) {
    if (int rc = check_raster(rs)) return rc;
    if (!pix_to_face || !zbuf || !bary || !dists) return PERT_E_NULL;
    if (rs->bin_faces && (!rs->bin_count || !rs->bin_offset)) return PERT_E_NULL;
    if (((uintptr_t)rs->bin_count & 3) || ((uintptr_t)rs->bin_offset & 7) || ((uintptr_t)rs->bin_faces & 7)) return PERT_E_ALIGN;
    if (((uintptr_t)pix_to_face & 7) || ((uintptr_t)zbuf & 3) || ((uintptr_t)bary & 3) || ((uintptr_t)dists & 3)) return PERT_E_ALIGN;
    return cuda_rc(launch_rasterize_fwd(*rs, pix_to_face, zbuf, bary, dists, (cudaStream_t)stream));
}

extern "C" int pert_rasterize_bwd(const pert_raster* rs, const int64_t* pix_to_face, const float* grad_zbuf,
                                  const float* grad_bary, const float* grad_dists, float* grad_face_verts, void* stream) {
    if (int rc = check_raster(rs)) return rc;
    if (!pix_to_face || !grad_face_verts) return PERT_E_NULL;
    if (((uintptr_t)pix_to_face & 7) || ((uintptr_t)grad_zbuf & 3) || ((uintptr_t)grad_bary & 3) || ((uintptr_t)grad_dists & 3) ||
        ((uintptr_t)grad_face_verts & 3))
        return PERT_E_ALIGN;
    return cuda_rc(launch_rasterize_bwd(*rs, pix_to_face, grad_zbuf, grad_bary, grad_dists, grad_face_verts, (cudaStream_t)stream));
}

extern "C" int64_t pert_rasterize_num_bins(const pert_raster* rs) {
    if (!rs || rs->N <= 0 || rs->H <= 0 || rs->W <= 0) return 0;
    return rs->N * (int64_t)((rs->W + 31) / 32) * (int64_t)((rs->H + 3) / 4);  // TW x TH tiles of csrc/raster.cu
}

extern "C" int pert_rasterize_bin(const pert_raster* rs, int32_t* bin_count, const int64_t* bin_offset, int32_t* bin_cursor,
                                  int64_t* bin_faces, void* stream) {
    if (int rc = check_raster(rs)) return rc;
    if (bin_faces ? (!bin_offset || !bin_cursor) : !bin_count) return PERT_E_NULL;
    if (((uintptr_t)bin_count & 3) || ((uintptr_t)bin_offset & 7) || ((uintptr_t)bin_cursor & 3) || ((uintptr_t)bin_faces & 7))
        return PERT_E_ALIGN;
    return cuda_rc(launch_rasterize_bin(*rs, bin_count, bin_offset, bin_cursor, bin_faces, (cudaStream_t)stream));
}
