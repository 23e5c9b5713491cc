/*
 * pertshade.h — C ABI of the B200-native perturbed shading hot path.
 *
 * One shared library (libpertshade.so, built for sm_100a from pertrenderer_b200/csrc) exports the
 * functions below.  Plain pointers and sizes only: no torch / C++ types cross this boundary, the
 * library never allocates, frees or retains device memory, never synchronises the device and launches on
 * the stream it is given.  The only state it keeps is diagnostic or immutable: the name of the calling thread's
 * last CUDA error (pert_last_cuda_error) and each device's SM count, cached at first use; it reads no environment
 * variable.  Every function returns PERT_OK (0) or a negative PERT_E_* code; nothing throws across the ABI.
 *
 * What each entry point replaces in the reference (paths relative to quentinll/pertrenderer):
 *
 *   pert_shade_fwd   randomras/random_rasterizer.py:34-56  smooth_rgb_blend          (forward), with
 *                    randomras/smoothrast.py:15-37         randomHeaviside.forward
 *                    randomras/smoothagg.py:196-205        GaussianAgg.aggregate
 *                    randomras/smoothagg.py:13-42          randomArgmax.forward
 *   pert_shade_bwd   the autograd backward of the same chain:
 *                    randomras/smoothagg.py:45-73          randomArgmax.backward
 *                    randomras/smoothagg.py:303-311,325-337 log_corrected / prod_corrected backward
 *                    randomras/smoothrast.py:40-59         randomHeaviside.backward
 *   pert_shade_render / pert_shade_render_phase   the forward of pert_shade_fwd (single call / one phase of a
 *                    sample-sharded call) when no gradient is wanted (torch.no_grad around smooth_rgb_blend)
 *   pert_soft_shade_fwd / _bwd        the same blend with SoftRast (smoothrast.py:126-134) + SoftAgg
 *                                     (smoothagg.py:165-182), the shaders' default operators
 *   pert_rast_fwd / pert_rast_bwd     randomras/smoothrast.py:12-59   (stand-alone randomHeaviside)
 *   pert_argmax_fwd / pert_argmax_bwd randomras/smoothagg.py:10-73    (stand-alone randomArgmax)
 *   pert_phong_fwd / pert_phong_bwd   pytorch3d.renderer.mesh.shading.phong_shading as called by
 *                    RandomPhongShader.forward (randomras/random_rasterizer.py:103-110), the shader
 *                    experiments/eval.py:170-176 uses; its output is the `colors` of pert_shade_fwd
 *   pert_rasterize_fwd / pert_rasterize_bwd   pytorch3d's MeshRasterizer -> rasterize_meshes as configured at
 *                    experiments/eval.py:135-141,165-169: the producer of the Fragments this path consumes
 *   pert_noise_fill  the two torch.normal draws, smoothrast.py:21 and smoothagg.py:21 (test aid:
 *                    materialises the counter-based noise the fused kernels generate in registers)
 *
 * Layouts (all contiguous, innermost last), P = N*H*W pixels, K faces per pixel, K1 = K+1:
 *   pix_to_face int64 (P,K)   zbuf, dists float (P,K)   colors float (P,K,3)
 *   znear, zfar float (N) or (1)   image / grad_image float (P,4)
 *   explicit noise: noise_rast float (S_rast,P,K), noise_agg float (S_agg,P,K1)   [optional]
 * Saved state written by forward and read by backward (caller-allocated):
 *   counts  uint16 (P,K)   number of coverage samples with h=1 among the local sample shard
 *   rsum    float  (P,K)   sum_s (h_s - h0) * U_s over the local sample shard
 *   winners uint8  (P,S_agg_local) if K1 <= 256 else uint16: argmax index of every sample; rows are
 *                  written only for pixels whose pixstate has the ACTIVE bit
 *   pixstate uint16 (P)    a0 | 0x8000 * active: a0 = unperturbed argmax (K = background), active =
 *                  some local sample picked another logit (inactive pixels: every sample picked a0)
 * Only entries with pix_to_face >= 0 are ever read or written in counts / rsum: real fragments are
 * sparse in K and the kernels touch zbuf / dists / saved state for valid entries only.
 */
#ifndef PERTSHADE_H_
#define PERTSHADE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PERT_ABI_VERSION 15

/* error codes */
#define PERT_OK 0
#define PERT_E_NULL (-1)        /* a required pointer is NULL */
#define PERT_E_SHAPE (-2)       /* non-positive / inconsistent sizes */
#define PERT_E_UNSUPPORTED (-3) /* K or S outside what the kernels support */
#define PERT_E_ALIGN (-4)       /* pointer not aligned to its element type */
#define PERT_E_SAMPLES (-5)     /* bad sample shard: begin must be a multiple of 4, begin < end <= S */
#define PERT_E_CUDA (-6)        /* CUDA launch / runtime error (see pert_last_cuda_error) */
#define PERT_E_SCALAR (-7)      /* sigma, gamma or alpha not finite and > 0 */

/* flags */
#define PERT_F_NO_SKIP 1u /* audit: no noise-bound based skipping (|x| > sigma*Umax entries, logits that
                             cannot win, radius gate, c_s = 0 quads); implies PERT_F_PER_SAMPLE_NOISE */
/* Backward, in-kernel (Philox) noise only.  A logit that can never win a sample (-inf, masked, or
 * further than 2*gamma*Umax below the largest) has noise V_sj independent of every winner a_s, so
 * given the c_s its score sum  sum_s c_s V_sj  is EXACTLY N(0, sum_s c_s^2).  Default: draw that
 * normal once per logit instead of S_agg times (same joint law of all gradients of dists / zbuf /
 * colors; the gamma-gradient's  sum_s c_s V_sj^2  keeps its mean and variance).
 *   PERT_F_PER_SAMPLE_NOISE: regenerate every V_sj of every logit instead, as the reference does
 *     (always the case with explicit noise): backward is then the explicit-noise kernel fed with
 *     pert_noise_fill's tensor, bit for bit.
 *   PERT_F_SKIP_DEAD_NOISE: replace those zero-mean terms by their expectation (0, and n*sum_s c_s
 *     for the squared term): same expectation, lower variance. */
#define PERT_F_SKIP_DEAD_NOISE 2u
#define PERT_F_PER_SAMPLE_NOISE 4u
/* standard Cauchy noise instead of Gaussian (ArctanRast smoothrast.py:162-173, CauchyAgg smoothagg.py:230-250): noise
 * tan(pi(u-1/2)) clamped to +-1e7, score 2n/(1+n^2) in backward.  Stand-alone operators, and pert_shade_fwd /
 * pert_shade_bwd with in-kernel or explicit noise, in one call or phase-split: there every valid entry draws all its
 * coverage samples, every finite logit takes part in the argmax and backward regenerates every V_sj of every logit
 * (the pert_noise_fill tensor of stage | 2 is the in-kernel stream).  The fused entry points return
 * PERT_E_UNSUPPORTED for PERT_F_CAUCHY with PERT_F_PHILOX7, PERT_F_NO_VR, PERT_F_SKIP_DEAD_NOISE, PERT_F_UNIFORM or
 * PERT_F_GUMBEL. */
#define PERT_F_CAUCHY 8u
/* Gaussian noise: the estimators WITHOUT the control variates, the paper's ablation
 * (randomHeaviside_wovr smoothrast.py:61-108: sum_s h_s U_s instead of sum_s (h_s - h0) U_s;
 *  randomArgmax_wovr smoothagg.py:75-141: c_s = <g, onehot(a_s)> instead of <g, onehot(a_s) - onehot(a_0)>).
 * Stand-alone operators, and pert_shade_fwd / pert_shade_bwd with in-kernel or explicit noise, in one call or
 * phase-split, with or without seed_device (GaussianRast_wovr + GaussianAgg_wovr).  Forward draws every coverage sample
 * of each valid entry with x >= -sigma*Umax (the others have h = 0 always) and has the per-sample path of
 * PERT_F_PER_SAMPLE_NOISE: counts, winners, image and alpha are those of the Gaussian pair with that flag, only rsum
 * differs.  Backward works on every valid pixel, including those whose samples all picked a_0 and those without any
 * valid entry (the background always wins; gamma term only), and regenerates every V_sj of every logit.  The fused
 * entry points return PERT_E_UNSUPPORTED for PERT_F_NO_VR with PERT_F_PHILOX7, PERT_F_SKIP_DEAD_NOISE, PERT_F_UNIFORM,
 * PERT_F_GUMBEL or PERT_F_CAUCHY.  Libraries older than pert_shade_fused_flags() ignore the flag in the fused entry
 * points: check that function before relying on it. */
#define PERT_F_NO_VR 0x400u
/* pert_argmax_fwd only: uniform noise on [-1/2, 1/2) (UniformAgg, smoothagg.py:252-272) or standard Gumbel noise
 * (randomArgmax "gumbel", smoothagg.py:22-24).  Forward only, as in the reference (no backward: smoothagg.py:64-67);
 * pert_argmax_bwd returns PERT_E_UNSUPPORTED with either flag. */
#define PERT_F_UNIFORM 0x800u
#define PERT_F_GUMBEL 0x1000u
/* pert_shade_fwd / pert_shade_bwd with in-kernel noise and all phases in one call: Philox4x32-7 instead of
 * Philox4x32-10 (7 rounds is the Crush-resistant minimum of Salmon et al., SC'11; 10 is their and cuRAND's default).
 * Another noise stream of the same law, 30 % fewer multiply / xor pairs per call; pert_noise_fill materialises it with
 * stage | 16.  Phase-split (sample-sharded) and explicit-noise calls return PERT_E_UNSUPPORTED with this flag. */
#define PERT_F_PHILOX7 0x2000u
/* phases of the fused kernels; 0 means "all".  Used for noise-sample sharding where collectives sit
 * between the phases (SURVEY.md §8e). */
#define PERT_PH_RAST 0x10u  /* fwd: draw coverage samples -> counts, rsum */
#define PERT_PH_AGG 0x20u   /* fwd: logits + perturbed argmax -> hist, winners   (reads counts if !RAST) */
#define PERT_PH_BLEND 0x40u /* fwd: hist -> image                                (reads hist if !AGG) */
#define PERT_PH_BWD_SAMPLE 0x100u /* bwd: per-logit score sums -> acc, pixstat */
#define PERT_PH_BWD_FINISH 0x200u /* bwd: chain rule -> grad_dists, grad_zbuf, scalars (reads acc if !SAMPLE) */

typedef struct pert_problem {
    /* geometry */
    int64_t N, H, W;
    int32_t K;
    /* hyper-parameters (GaussianRast.sigma, GaussianAgg.gamma/.alpha/.eps, BlendParams.background_color) */
    float sigma, gamma, alpha, eps;
    float background[3];
    /* sample counts: totals are the estimator's denominators; [begin,end) is this call's shard */
    int32_t S_rast, S_agg;
    int32_t s_rast_begin, s_rast_end;
    int32_t s_agg_begin, s_agg_end;
    /* counter-based noise: seeds of the two stages, global index of this call's first pixel */
    uint64_t seed_rast, seed_agg;
    int64_t pixel_offset;
    uint32_t flags;
    int32_t depth_len; /* length of znear/zfar: 1 (broadcast) or N */
    /* inputs (device pointers) */
    const int64_t* pix_to_face;
    const float* zbuf;
    const float* dists;
    const float* colors;
    const float* znear;
    const float* zfar;
    /* optional explicit noise (device); NULL -> in-register Philox4x32-10 + Box-Muller */
    const float* noise_rast;
    const float* noise_agg;
    /* optional per-face colours float (num_faces,3): when set, `colors` is ignored (may be NULL) and the
     * colour of entry (p,k) is face_colors[pix_to_face[p,k]] gathered inside the kernels — the (P,K,3)
     * texel tensor of Meshes.sample_textures (random_rasterizer.py:170) is never materialised */
    const float* face_colors;
    int64_t num_faces;
    /* optional device-side seeds, uint64[2] (device) or NULL: when set the fused kernels draw with seed_rast ^ seed_device[0]
     * and seed_agg ^ seed_device[1], read at launch.  A forward + backward pair captured in a CUDA graph (together with a
     * pert_seed_advance node) then draws fresh noise at every replay although every launch parameter is frozen: the
     * small-problem path, where launch overhead dominates (experiments/eval.py:341-394 loops over 64x64..128x128 images) */
    const uint64_t* seed_device;
} pert_problem;

int pert_version(void);
/* PERT_F_* estimator / noise flags that pert_shade_fwd / pert_shade_bwd implement (PERT_F_CAUCHY, PERT_F_NO_VR, ...).
 * A flag that is not in this set is rejected or ignored by the fused entry points of this library; callers check a
 * flag here before its first fused call, so that an older library is detected rather than silently ignoring it. */
uint32_t pert_shade_fused_flags(void);
const char* pert_strerror(int code);
/* last cudaError_t name seen by this thread's most recent failing call (diagnostic only) */
const char* pert_last_cuda_error(void);

/* number of warp tiles (= CTAs) T the fused kernels launch.  Workspaces (caller-allocated, 16-byte aligned):
 *   scalar_partials  float  4 * 3T   (one row per tile; rows T..3T belong to the fallback pass)
 *   worklist         int32  4 + T    optional (NULL: off).  Sparse-first mode: the main pass holds half a
 *                    tile's entries in shared memory (real fragments fill a few percent); tiles with more
 *                    valid entries are listed here and redone by a fallback pass as half-size tiles (forward:
 *                    two launches, coverage samples then aggregation + blend).  Words 0..3 are the list length
 *                    and the work cursors of the fallback launches, words 4.. the tile ids; the library zeroes
 *                    the header itself (cudaMemsetAsync on the caller's stream).  Results do not depend on
 *                    which pass handled a tile, up to the association order of float sums. */
int64_t pert_num_tiles(const pert_problem* pb);
/* element size in bytes of the winners buffer for this K (1 or 2) */
int pert_winner_bytes(int32_t K);
/* size in bytes of the optional `tile_blob` buffer (16-byte aligned).  In sparse-first mode forward saves,
 * per warp tile, the compact list of valid entries and the per-pixel logit summary it computed, for the tiles of
 * the main pass and for the half-tiles of the fallback pass (room for every tile to take the fallback pass: at
 * 8 x 256^2, K = 50, 57 MB of tile blobs and 173 MB of fallback records); backward then neither re-scans
 * pix_to_face nor recomputes the logits, and the second forward launch of the fallback pass does not re-scan.
 * Pass the SAME flags / geometry to both calls.  NULL: both recompute (same results). */
int64_t pert_blob_bytes(const pert_problem* pb);

/*
 * Forward.  Outputs: image (P,4).  Saved state: counts, rsum, winners, pixstate (see top).  `hist` int32
 * (P,K1) is optional unless the AGG and BLEND phases run in separate calls.  With phase flags,
 * buffers produced by an earlier phase are inputs.
 */
int pert_shade_fwd(const pert_problem* pb, float* image, uint16_t* counts, float* rsum, void* winners,
                   uint16_t* pixstate, int32_t* hist, int32_t* worklist, void* tile_blob, void* stream);

/*
 * Forward-only render: the image of pert_shade_fwd for a call that needs no gradient (evaluation renders, high sample
 * counts).  Nothing is stored for backward: no counts, rsum, winners, pixstate or tile blob.  Coverage computes hit
 * counts only (the compound sampler draws the number of flips and no tail normals, the per-sample path keeps its h
 * tests and drops the score sums), from the same counters as pert_shade_fwd, and the winner histogram stays in shared
 * memory.  For the same problem (seeds, flags, noise) the image equals pert_shade_fwd's bit for bit, and no buffer
 * depends on S_rast or S_agg.  Same flags and flag rules as pert_shade_fwd (PERT_F_CAUCHY, PERT_F_NO_VR, PERT_F_PHILOX7,
 * explicit noise, face_colors, pixel_offset, seed_device); single calls only: any PERT_PH_* bit, or a sample shard
 * other than [0, S), returns PERT_E_UNSUPPORTED.  Workspaces (caller-allocated):
 *   worklist   int32 4 + pert_num_tiles, 16-byte aligned, optional (NULL: sparse-first mode off), as in pert_shade_fwd
 *   counts_ws  uint16 (P,K), required when the sparse-first mode can run (worklist set, in-kernel Gaussian noise without
 *              PERT_F_NO_SKIP / PER_SAMPLE_NOISE / CAUCHY / NO_VR): its fallback pass runs as two launches and keeps the
 *              counts of its tiles here between them.  Unused (may be NULL) otherwise
 */
int pert_shade_render(const pert_problem* pb, float* image, uint16_t* counts_ws, int32_t* worklist, void* stream);

/*
 * Forward-only render of one phase of the sample-sharded (phase-split) forward: pb->flags carries exactly one of
 * PERT_PH_RAST, PERT_PH_AGG and PERT_PH_BLEND, and [s_rast_begin, s_rast_end) / [s_agg_begin, s_agg_end) are this call's
 * sample shards.  Nothing is stored for backward and no buffer depends on S_rast or S_agg:
 *   PERT_PH_RAST   writes the shard's hit counts to `counts` (uint16 (P,K)) at the entries with pix_to_face >= 0 only;
 *                  padding entries are left as they are (zero the buffer before summing it over shards)
 *   PERT_PH_AGG    reads the all-shard `counts`, writes every entry of `hist` (int32 (P,K1)): the shard's winner histogram
 *   PERT_PH_BLEND  reads `counts` (alpha) and the all-shard `hist`, writes `image`
 * For the same problem and phase the outputs equal those of pert_shade_fwd bit for bit.  Flag rules are pert_shade_render's
 * (PERT_F_CAUCHY, PERT_F_NO_VR, explicit noise, face_colors, pixel_offset, seed_device), except that PERT_F_PHILOX7 is
 * refused, as in every phase-split call.  No phase bit, several, or a PERT_PH_BWD_* bit returns PERT_E_UNSUPPORTED.
 */
int pert_shade_render_phase(const pert_problem* pb, float* image, uint16_t* counts, int32_t* hist, void* stream);

/*
 * Backward.  grad_image (P,4).  Outputs grad_dists, grad_zbuf (P,K), grad_colors (P,K,3; may be
 * NULL), grad_scalars float[3] = d/d(sigma, gamma, alpha).  With pb->face_colors set, grad_colors is
 * instead float (num_faces,3), ZEROED BY THE CALLER, and receives w_k * dL/drgb by atomic adds (the
 * scatter of Meshes.sample_textures' backward; summation order is not fixed).  scalar_partials: workspace of
 * 4*pert_num_tiles floats.  acc float (P,K1) and pixstat float (P,2) are optional unless the two
 * backward phases run in separate calls (sample sharding); hist int32 (P,K1) is the all-shard
 * winner histogram of forward, needed only then (NULL: rebuilt from `winners` / `pixstate`).
 */
int pert_shade_bwd(const pert_problem* pb, const float* grad_image, const uint16_t* counts,
                   const float* rsum, const void* winners, const uint16_t* pixstate, float* grad_dists,
                   float* grad_zbuf, float* grad_colors, float* scalar_partials, float* grad_scalars,
                   float* acc, float* pixstat, const int32_t* hist, int32_t* worklist, const void* tile_blob,
                   void* stream);

/*
 * SoftRas pair: SoftRast + SoftAgg, the DEFAULT operators of RandomSimpleShader
 * (randomras/random_rasterizer.py:139-140; smoothrast.py:126-134; smoothagg.py:165-182), fused and
 * deterministic: P = sigmoid(-dists/sigma)*mask, w = softmax(logits/gamma), same logits, alpha channel and
 * blend as the perturbed shader.  The sample-count / seed / noise fields of pert_problem are ignored.
 * Backward recomputes forward (no saved state): outputs as pert_shade_bwd, scalar_partials needs
 * 4 * pert_num_tiles floats.
 */
int pert_soft_shade_fwd(const pert_problem* pb, float* image, void* stream);
int pert_soft_shade_bwd(const pert_problem* pb, const float* grad_image, float* grad_dists, float* grad_zbuf,
                        float* grad_colors, float* scalar_partials, float* grad_scalars, void* stream);

/*
 * Stand-alone perturbed Heaviside on x (P,K) (x = -dists in the shader).  prob = counts/S.
 * Explicit noise (S,P,K) optional.
 */
int pert_rast_fwd(const float* x, int64_t P, int32_t K, int32_t S, int32_t s_begin, int32_t s_end,
                  float sigma, uint64_t seed, int64_t pixel_offset, const float* noise, uint32_t flags,
                  float* prob, float* rsum, void* stream);
int pert_rast_bwd(const float* grad_l, const float* rsum, int64_t n, int32_t S, float sigma,
                  float* grad_x, float* scalar_partials, float* grad_sigma, void* stream);

/* Stand-alone perturbed argmax on logits z (P,K1). */
int pert_argmax_fwd(const float* z, int64_t P, int32_t K1, int32_t S, int32_t s_begin, int32_t s_end,
                    float gamma, uint64_t seed, int64_t pixel_offset, const float* noise, uint32_t flags,
                    float* weights, void* winners, void* stream);
int pert_argmax_bwd(const float* grad_l, const float* z, const void* winners, int64_t P, int32_t K1,
                    int32_t S, int32_t s_begin, int32_t s_end, float gamma, uint64_t seed,
                    int64_t pixel_offset, const float* noise, uint32_t flags, float* grad_z,
                    float* scalar_partials, float* grad_gamma, void* stream);

/*
 * Phong lighting of every fragment entry: the `colors` (P,K,3) that RandomPhongShader feeds to
 * smooth_rgb_blend (randomras/random_rasterizer.py:103-113).  Restates pytorch3d 0.4.0 (requirements.txt:7;
 * source not part of the reference tree): shading.phong_shading -> interpolate_face_attributes of the face
 * corners' positions and vertex normals with bary_coords, lighting.diffuse / lighting.specular of a
 * PointLights or DirectionalLights, Materials, colour = (ambient + diffuse) * texel + specular.
 *
 * `lighting`: float (light_rows, PERT_PHONG_STRIDE), one row per batch element (or one row for all):
 *   [0:3] light location (point) or direction (directional)   [3:6]  materials.ambient * lights.ambient
 *   [6:9] materials.diffuse * lights.diffuse                  [9:12] materials.specular * lights.specular
 *   [12]  materials.shininess   [13:16] camera centre (world)  [16]  0 = point light, 1 = directional
 * Entries with pix_to_face < 0 interpolate to a zero point and normal (pytorch3d's masked interpolation), so
 * their colour is ambient * texel.  With PERT_PHONG_SPARSE those entries are skipped altogether: forward does
 * not write their colour (the fused shader kernels never read it), backward neither reads their grad_colors
 * (the fused shader's is 0 there) nor writes their grad_texels / grad_bary (pre-zero them if they are read).
 */
#define PERT_PHONG_STRIDE 20
#define PERT_PHONG_SPARSE 1u
/* texture sampling only: colour = texel, no lighting (face_verts / face_normals / lighting may be NULL).  With
 * face_vert_colors this is TexturesVertex.sample_textures (interpolate_face_attributes of the vertex colours,
 * experiments/eval.py:450), with face_colors a per-face colour lookup: Meshes.sample_textures at
 * randomras/random_rasterizer.py:101,170 without leaving the kernels' sparse entry lists. */
#define PERT_PHONG_UNLIT 2u

typedef struct pert_phong {
    int64_t P;          /* pixels N*H*W */
    int64_t HW;         /* pixels per batch element: selects the lighting row */
    int32_t K;
    int32_t light_rows; /* 1 or N */
    int64_t num_faces;
    uint32_t flags;
    const int64_t* pix_to_face; /* (P,K) */
    const float* bary;          /* (P,K,3) fragments.bary_coords */
    const float* face_verts;    /* (F,3,3) verts_packed()[faces_packed()] */
    const float* face_normals;  /* (F,3,3) verts_normals_packed()[faces_packed()] */
    const float* texels;        /* (P,K,3) meshes.sample_textures(fragments), or NULL with face_colors */
    const float* face_colors;   /* (F,3) per-face colours gathered through pix_to_face, or NULL */
    const float* lighting;      /* (light_rows, PERT_PHONG_STRIDE) */
    const float* face_vert_colors; /* (F,3,3) colours at the face corners, interpolated with bary (TexturesVertex:
                                      verts_features_packed()[faces_packed()]), or NULL */
    /* UV texture (TexturesUV / the legacy Textures of experiments/eval.py:750-756), or NULL: the texel is the bilinear
     * tap (grid_sample: align_corners, border padding, map flipped vertically) of uv_map at sum_i bary_i * face_uvs[f,i] */
    const float* face_uvs;  /* (F,3,2) verts_uvs[faces_uvs] */
    const float* uv_map;    /* (map_count, map_h, map_w, 3), map_count = 1 or N (one map per image) */
    int32_t map_h, map_w, map_count;
    int64_t faces_per_mesh; /* optional hint, 0 = none: the faces are N equal ranges, image n using only faces
                               [n * faces_per_mesh, (n+1) * faces_per_mesh) (a batch of poses of one topology); lets
                               backward keep one shared-memory gradient table per image.  Results do not depend on it */
} pert_phong;

int pert_phong_fwd(const pert_phong* ph, float* colors, void* stream);
/*
 * Backward of pert_phong_fwd.  grad_colors (P,K,3).  Outputs, each optional (NULL: not computed):
 *   grad_texels        (P,K,3); with ph->face_colors set: (F,3), with ph->face_vert_colors set: (F,3,3), with ph->uv_map set:
 *                      the map's shape; these three ZEROED BY THE CALLER, atomic adds (face_uvs gets no gradient)
 *   grad_bary          (P,K,3)
 *   grad_face_verts    (F,3,3) and grad_face_normals (F,3,3): ZEROED BY THE CALLER, atomic adds (the scatter of
 *                      interpolate_face_attributes' backward; summation order is not fixed)
 *   grad_lighting      (light_rows, PERT_PHONG_STRIDE), ZEROED BY THE CALLER: gradient of the lighting table (columns
 *                      0:16: light location / direction, the three colour products, shininess, camera centre), for
 *                      callers that optimise lights or cameras (experiments/eval.py:411-470, 693-725); a second sparse pass
 */
int pert_phong_bwd(const pert_phong* ph, const float* grad_colors, float* grad_texels, float* grad_bary,
                   float* grad_face_verts, float* grad_face_normals, float* grad_lighting, void* stream);

/*
 * Phong with a per-face texture atlas as the texel source (pytorch3d TexturesAtlas, the ShapeNet models of
 * experiments/eval.py:216-238): atlas float (ph->num_faces, R, R, 3), R = atlas_size, indexed by the packed face id.  The
 * texel of a valid entry is the atlas cell that its first two barycentric coordinates w0, w1 pick, in float32:
 *   w   = torch.nan_to_num(w, nan=0): NaN -> 0, +-inf -> +-FLT_MAX (both coordinates)
 *   wxy = trunc(clamp(w * R, -1, R)), then at most R - 1
 *   below = (w0 + w1) * R - (wx + wy) <= 1     (each operation rounded once, no fused multiply-add)
 *   (wx, wy) = below ? (wx, wy) : (R - 1 - wx, R - 1 - wy), then clamped to [0, R - 1]
 *   texel = atlas[face, wy, wx]
 * which is AtlasTexels.materialize (pertrenderer_b200/structures.py).  Padded entries get texel 0.  Everything else
 * (flags, lighting, sparse / unlit modes, validation) is pert_phong_fwd / pert_phong_bwd's, except the texel source:
 * ph->texels, face_colors, face_vert_colors and uv_map must all be NULL (else PERT_E_UNSUPPORTED); a NULL atlas returns
 * PERT_E_NULL, atlas_size <= 0 PERT_E_SHAPE, and num_faces * R^2 * 3 > 2^31 - 1 (32-bit atlas offsets) PERT_E_UNSUPPORTED.
 * Neither call synchronises: both can be captured in a CUDA graph.
 */
int pert_phong_atlas_fwd(const pert_phong* ph, const float* atlas, int32_t atlas_size, float* colors, void* stream);
/*
 * Backward of pert_phong_atlas_fwd.  Outputs as pert_phong_bwd's, each optional (NULL: not computed), with grad_atlas in
 * the place of grad_texels: the atlas's shape, ZEROED BY THE CALLER, the texel gradient atomically added into the cell of
 * every entry (summation order is not fixed).  The atlas texel is piecewise constant in the barycentric coordinates, so
 * it adds nothing to grad_bary: lit entries get the gradient of their position and normal only, unlit entries zero.
 */
int pert_phong_atlas_bwd(const pert_phong* ph, const float* atlas, int32_t atlas_size, const float* grad_colors,
                         float* grad_atlas, float* grad_bary, float* grad_face_verts, float* grad_face_normals,
                         float* grad_lighting, void* stream);

/*
 * Fragment producer: K-deep rasterisation of packed triangle meshes with a blur radius, the Fragments
 * (pix_to_face, zbuf, bary_coords, dists) of pytorch3d's MeshRasterizer as the reference configures it
 * (experiments/eval.py:135-141: blur_radius = log(1/1e-4 - 1) * sigma, faces_per_pixel = 50,
 * perspective_correct = False, no barycentric clipping).  Restates pytorch3d 0.4.0's naive rasteriser
 * (rasterize_meshes.cu CheckPixelInsideFace, geometry_utils.cuh, kEpsilon = 1e-8); see csrc/raster.cu.
 *
 * face_verts float (F,3,3): per face corner NDC x, NDC y (+X left, +Y up; pixel (0,0) is the top-left corner) and
 * VIEW-space depth z, as MeshRasterizer.transform produces them.  face_start int64 (N+1), device: the faces
 * [face_start[n], face_start[n+1]) are rasterised into image n.  Outputs, all written in full (padding -1):
 * pix_to_face int64 (N,H,W,K) packed face index, zbuf float (N,H,W,K) ascending (ties in face order), bary float
 * (N,H,W,K,3), dists float (N,H,W,K) signed squared NDC distance to the face (negative inside).
 */
#define PERT_RAST_CULL_BACKFACES 1u
/* the rs->bin_* lists are the bounded layout of pert_rasterize_bin_bounded (num_bins + N bins; the last N are the
 * images' wide lists).  Requires rs->bin_faces (else PERT_E_NULL) */
#define PERT_RAST_BIN_WIDE 2u

typedef struct pert_raster {
    int64_t N;
    int32_t H, W, K;
    uint32_t flags;
    float blur_radius;
    int64_t num_faces;
    const float* face_verts;   /* (F,3,3) */
    const int64_t* face_start; /* (N+1), device */
    const int64_t* face_order; /* optional (F): a permutation of every range [face_start[n], face_start[n+1]) giving the
                                  order in which the faces are visited.  The result does not depend on it (the K-buffer
                                  is ranked at the end); kept for callers that want a traversal order.  NULL: index
                                  order.  Forward, K <= 64 only */
    /* optional coarse bins (forward, K <= 64): one list of candidate faces per 32x4 pixel tile, built by two
     * pert_rasterize_bin calls; every tile then walks its own list instead of all faces of its mesh.  For meshes of
     * thousands of faces.  NULL: off.  With PERT_RAST_BIN_WIDE, the bounded layout of pert_rasterize_bin_bounded:
     * N * tiles + N bins, every tile walking its own list and then its image's wide list */
    const int32_t* bin_count;  /* (N * tiles [+ N]) faces per tile, tiles = ceil(W/32) * ceil(H/4) */
    const int64_t* bin_offset; /* (N * tiles [+ N]) start of every list in bin_faces: exclusive prefix sum of bin_count */
    const int64_t* bin_faces;  /* (sum of bin_count) packed face indices */
} pert_raster;

/* number of bins of this problem: N * ceil(W/32) * ceil(H/4) */
int64_t pert_rasterize_num_bins(const pert_raster* rs);
/*
 * Coarse binning, two calls around an exclusive prefix sum done by the caller:
 *   1. bin_faces = NULL: counts the candidate faces of every tile into bin_count (int32, ZEROED BY THE CALLER)
 *   2. bin_faces != NULL: with bin_offset = exclusive prefix sum of bin_count and bin_cursor (int32, ZEROED BY THE
 *      CALLER), writes every tile's list; bin_faces holds sum(bin_count) entries.
 * The rs->bin_* fields are ignored here.
 */
int pert_rasterize_bin(const pert_raster* rs, int32_t* bin_count, const int64_t* bin_offset, int32_t* bin_cursor,
                       int64_t* bin_faces, void* stream);
/*
 * Coarse binning whose total length is known on the host, so that nothing is read back between the two calls (a CUDA
 * graph can capture them).  A face whose grown bounding box overlaps at most C tiles (C, a compile-time constant: 8)
 * is listed in those tiles, as by pert_rasterize_bin; a face overlapping more (a box reaching +-inf or NaN covers the
 * whole axis) is listed once in the WIDE list of its image, which every tile of that image walks too.  The arrays hold
 * pert_rasterize_num_bins(rs) + N entries: the tile bins, then the wide lists of images 0..N-1.  The two calls and
 * their rules are those of pert_rasterize_bin; bin_faces needs at most pert_rasterize_bin_capacity(rs) entries.  The
 * forward reads the result with rs->flags |= PERT_RAST_BIN_WIDE.
 */
int pert_rasterize_bin_bounded(const pert_raster* rs, int32_t* bin_count, const int64_t* bin_offset, int32_t* bin_cursor,
                               int64_t* bin_faces, void* stream);
/* upper bound of the total length of pert_rasterize_bin_bounded's lists: C * num_faces (0 for a NULL or empty problem) */
int64_t pert_rasterize_bin_capacity(const pert_raster* rs);

int pert_rasterize_fwd(const pert_raster* rs, int64_t* pix_to_face, float* zbuf, float* bary, float* dists, void* stream);
/*
 * Backward of pert_rasterize_fwd (rasterize_meshes' autograd backward): gradients of zbuf (N,H,W,K), bary
 * (N,H,W,K,3) and dists (N,H,W,K), each optional (NULL = zero), to grad_face_verts float (F,3,3), ZEROED BY THE
 * CALLER, atomic adds.
 */
int pert_rasterize_bwd(const pert_raster* rs, const int64_t* pix_to_face, const float* grad_zbuf, const float* grad_bary,
                       const float* grad_dists, float* grad_face_verts, void* stream);

/* Advance device-side seeds (pert_problem.seed_device): seed_device[i] <- splitmix64 step of seed_device[i], i = 0, 1.  One
 * single-thread launch on `stream`; capturable in a CUDA graph. */
int pert_seed_advance(uint64_t* seed_device, void* stream);

/* Materialise the counter-based noise: out float (s_end-s_begin, P, slots), stage 0 = coverage
 * (slots = K), 1 = aggregation (slots = K1); stage | 2 = the Cauchy variant of that stage, | 4 uniform, | 8 Gumbel,
 * | 16 the Gaussian stream of PERT_F_PHILOX7. */
int pert_noise_fill(uint64_t seed, int32_t stage, int64_t P, int32_t slots, int32_t s_begin, int32_t s_end,
                    int64_t pixel_offset, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PERTSHADE_H_ */
