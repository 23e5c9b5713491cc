// Phong lighting of the fragment entries (pert_phong_fwd / pert_phong_bwd in include/pertshade.h): the
// `colors` (P,K,3) RandomPhongShader hands to smooth_rgb_blend (randomras/random_rasterizer.py:103-113).
//
// Restates pytorch3d 0.4.0 (requirements.txt:7; its source is not under the reference tree):
//   shading.phong_shading:      pixel_coords / pixel_normals = interpolate_face_attributes(pix_to_face, bary, .)
//                               colors = (ambient + diffuse) * texels + specular
//   shading._apply_lighting:    ambient = materials.ambient * lights.ambient, diffuse = materials.diffuse *
//                               lights.diffuse(normals, points), specular = materials.specular * lights.specular(..)
//   lighting.diffuse/specular:  F.normalize(., eps=1e-6) of normal, light direction and view direction,
//                               relu(n.d), reflect = -d + 2 (n.d) n, relu(v.r) * [n.d > 0], pow(., shininess)
//
// A streaming pass over the (P,K) entries: pix_to_face is read coalesced (8 B per entry); everything else is
// touched for valid entries only (real fragments are sparse in K), and in backward only for entries whose
// colour gradient is non-zero (the blend gives weight to a few winners per pixel).  The entries that need the
// lighting arithmetic are compacted per warp so that full warps execute it.  Face-table gradients go
// through a per-CTA shared-memory table when the mesh is small (every CTA would hammer the same few hundred
// L2 addresses otherwise) and straight to global atomics when it is large.
#include "kernels.h"
#include "texel.cuh"
#include "tile.cuh"

namespace pert {

namespace {

constexpr int PT = 128;  // threads per CTA (forward, and backward without a shared-memory gradient table)
constexpr int PW = PT / 32;
constexpr int PT_TABLE = 512;  // backward with the gradient table: ONE CTA per SM, 16 warps sharing the table (24 warps at an
                               // 80-register cap were slower: 273 vs 238 us)
constexpr int WCHUNK = 1024;  // entries a warp scans at a time
constexpr int TABLE_MAX_BYTES = 150 * 1024;  // table of 18..27 floats per face (F <= 2133..1422) next to 66 KB of warp lists

constexpr float kNormEps = 1e-6f;  // F.normalize(eps=1e-6) in pytorch3d's lighting.py

// x = raw / max(|raw|, eps)
__device__ __forceinline__ V3 normalize(V3 raw, float& len) {
    len = sqrtf(dot(raw, raw));
    return (1.0f / fmaxf(len, kNormEps)) * raw;
}
// gradient of normalize: (g - x (x.g)) / |raw| where the clamp is inactive, g / eps where it is
__device__ __forceinline__ V3 normalize_bwd(V3 x, float len, V3 g) {
    if (len > kNormEps) return (1.0f / len) * (g - dot(x, g) * x);
    return (1.0f / kNormEps) * g;
}

struct Row {  // one row of `lighting`
    V3 loc, amb, dif, spc, cam;
    float sh;
    bool directional;
};
__device__ __forceinline__ Row row_from(const float* r) {
    Row o;
    o.loc = mk(r[0], r[1], r[2]);
    o.amb = mk(r[3], r[4], r[5]);
    o.dif = mk(r[6], r[7], r[8]);
    o.spc = mk(r[9], r[10], r[11]);
    o.sh = r[12];
    o.cam = mk(r[13], r[14], r[15]);
    o.directional = r[16] != 0.0f;
    return o;
}

struct Lit {  // what backward needs of the forward evaluation
    V3 n, d, v, r;
    float nl, dl, vl, cosd, ang, vr, alpha, pw;
};

__device__ __forceinline__ Lit light_entry(const Row& L, V3 p, V3 n_raw) {
    Lit o;
    o.n = normalize(n_raw, o.nl);
    o.d = normalize(L.directional ? L.loc : L.loc - p, o.dl);
    o.cosd = dot(o.n, o.d);
    o.ang = fmaxf(o.cosd, 0.0f);
    o.v = normalize(L.cam - p, o.vl);
    o.r = (2.0f * o.cosd) * o.n - o.d;
    o.vr = dot(o.v, o.r);
    o.alpha = o.cosd > 0.0f ? fmaxf(o.vr, 0.0f) : 0.0f;
    o.pw = powf(o.alpha, L.sh);
    return o;
}


// Texel of a valid entry from whichever source the call carries: the caller's (P,K,3) tensor, one colour per face
// (F,3), colours at the face corners (F,3,3) interpolated with the barycentric coordinates (TexturesVertex), or a UV
// map sampled at the interpolated corner UVs (TexturesUV; the `Textures(verts_uvs, faces_uvs, maps)` of
// experiments/eval.py:750-756).
__device__ __forceinline__ V3 texel_of_plain(const pert_phong& ph, int64_t e, int64_t face, V3 b) {
    if (ph.face_vert_colors) return vert_texel(ph.face_vert_colors + face * 9, b);
    return ph.face_colors ? ld3(ph.face_colors + face * 3) : ld3(ph.texels + e * 3);
}
__device__ __forceinline__ V3 texel_of(const pert_phong& ph, int64_t e, int64_t face, V3 b) {
    if (ph.uv_map) return uv_texel(uv_src(ph), e, face, b);
    return texel_of_plain(ph, e, face, b);
}
// Texel of the call's source: the atlas in the ATLAS instantiations, else texel_of
template <bool ATLAS>
__device__ __forceinline__ V3 texel_src(const pert_phong& ph, AtlasSrc at, int64_t e, int64_t face, V3 b) {
    if (ATLAS) return atlas_texel(at, face, b);
    return texel_of(ph, e, face, b);
}

// floats per face of the texel source's gradient table (0: dense (P,K,3) gradient, or the UV map's own gradient)
__host__ __device__ __forceinline__ int tex_floats(const pert_phong& ph) {
    return ph.uv_map ? 0 : (ph.face_vert_colors ? 9 : (ph.face_colors ? 3 : 0));
}

// The lighting rows of the batch elements a chunk of entries can touch: the chunk's first batch element and
// the next one sit in (per-warp) shared memory, anything further (tiny images) is read from global memory.
struct RowCache {
    const float* s;  // 2 * PERT_PHONG_STRIDE floats
    int64_t b0;
    const float* g;
    __device__ __forceinline__ Row get(int64_t b) const {
        const int64_t o = b - b0;
        if (o == 0 || o == 1) return row_from(s + o * PERT_PHONG_STRIDE);
        float r[PERT_PHONG_STRIDE];
#pragma unroll
        for (int i = 0; i < 17; ++i) r[i] = __ldg(g + b * PERT_PHONG_STRIDE + i);
        return row_from(r);
    }
};

__device__ __forceinline__ void fill_rows(const pert_phong& ph, int64_t b0, float* srow, int lane) {
    const int64_t nb = ph.light_rows;
    for (int i = lane; i < 2 * PERT_PHONG_STRIDE; i += 32) {
        const int64_t b = b0 + i / PERT_PHONG_STRIDE;
        srow[i] = __ldg(ph.lighting + (b < nb ? b : nb - 1) * PERT_PHONG_STRIDE + i % PERT_PHONG_STRIDE);
    }
}

// Warp-autonomous chunks (no block-level synchronisation in the streaming loop): a warp scans WCHUNK
// consecutive entries of pix_to_face with 128-bit loads and compacts the valid ones into its own shared list
// (scan_valid of tile.cuh, the scan of the fused shader kernels), then full warps walk the list.  Without the
// compaction a warp of 32 consecutive entries holds 2-3 valid ones on real fragments and the lighting code runs
// at 8 of 32 lanes (measured: 7.9 threads per instruction, r3a); with CTA-wide phases and barriers the kernel was
// latency-bound (r3b).
struct WarpCtx {
    int lane, warp;
    uint16_t* vlist;  // WCHUNK
    uint16_t* hlist;  // WCHUNK (backward: the entries with a non-zero colour gradient)
    float* srow;      // 2 * PERT_PHONG_STRIDE
};

template <bool ATLAS>
__global__ void __launch_bounds__(PT) phong_fwd_kernel(const pert_phong ph, float* __restrict__ colors, int64_t E,
                                                       int64_t nchunks, int vec_ok, AtlasSrc at) {
    __shared__ __align__(16) uint16_t s_vlist[PW][WCHUNK];
    __shared__ float s_row[PW][2 * PERT_PHONG_STRIDE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t* const vlist = s_vlist[warp];
    float* const srow = s_row[warp];
    const bool sparse = ph.flags & PERT_PHONG_SPARSE, unlit = ph.flags & PERT_PHONG_UNLIT;
    const bool table_tex = ATLAS || ph.face_colors || ph.face_vert_colors || ph.uv_map;
    const int64_t HWK = ph.HW * ph.K;
    int64_t cached_b0 = -1;
    const int64_t w0 = (int64_t)blockIdx.x * PW + warp, wstride = (int64_t)gridDim.x * PW;
#pragma unroll 1
    for (int64_t c = w0; c < nchunks; c += wstride) {
        const int64_t e_base = c * WCHUNK;
        const int Ec = (int)min((int64_t)WCHUNK, E - e_base);
        const int64_t b0 = ph.light_rows > 1 ? e_base / HWK : 0;
        if (b0 != cached_b0 && !unlit) {  // warp-uniform
            __syncwarp();
            fill_rows(ph, b0, srow, lane);
            cached_b0 = b0;
        }
        const RowCache rows{srow, b0, ph.lighting};
        const int64_t* const p2f = ph.pix_to_face + e_base;
        const int nv = scan_valid(p2f, Ec, vec_ok, vlist, WCHUNK);
        __syncwarp();
        if (!sparse && nv < Ec) {
            // masked interpolation: zero point and normal -> no diffuse, alpha = 0; what is left is
            // ambient * texel (+ specular * 0^shininess, which is 1 for shininess 0)
#pragma unroll 1
            for (int i = lane; i < Ec; i += 32) {
                if (__ldg(p2f + i) >= 0) continue;
                const int64_t e = e_base + i;
                const Row L = rows.get(ph.light_rows > 1 ? e / HWK : 0);
                const V3 t = table_tex ? mk(0.f, 0.f, 0.f) : ld3(ph.texels + e * 3);
                const float pw = L.sh == 0.0f ? 1.0f : 0.0f;
                st3(colors + e * 3, unlit ? t : mk(L.amb.x * t.x + L.spc.x * pw, L.amb.y * t.y + L.spc.y * pw, L.amb.z * t.z + L.spc.z * pw));
            }
        }
#pragma unroll 1
        for (int i = lane; i < nv; i += 32) {
            const int64_t e = e_base + vlist[i];
            const int64_t face = __ldg(ph.pix_to_face + e);
            const V3 b = ld3(ph.bary + e * 3);
            const V3 t = texel_src<ATLAS>(ph, at, e, face, b);
            if (unlit) {  // texture sampling only (Meshes.sample_textures)
                st3(colors + e * 3, t);
                continue;
            }
            const float* fv = ph.face_verts + face * 9;
            const float* fn = ph.face_normals + face * 9;
            const V3 p = b.x * ld3(fv) + b.y * ld3(fv + 3) + b.z * ld3(fv + 6);
            const V3 nr = b.x * ld3(fn) + b.y * ld3(fn + 3) + b.z * ld3(fn + 6);
            const Row L = rows.get(ph.light_rows > 1 ? e / HWK : 0);
            const Lit o = light_entry(L, p, nr);
            st3(colors + e * 3, mk((L.amb.x + L.dif.x * o.ang) * t.x + L.spc.x * o.pw,
                                   (L.amb.y + L.dif.y * o.ang) * t.y + L.spc.y * o.pw,
                                   (L.amb.z + L.dif.z * o.ang) * t.z + L.spc.z * o.pw));
        }
        __syncwarp();
    }
}

// TABLE: accumulate the (F,3,3) gradients of face_verts / face_normals (and the (F,3) gradient of
// face_colors) in shared memory and flush once per CTA.
// dst[3 i + c] += b_i * g_c for the three corners: into the shared-memory table or into global memory.  Two separate
// code paths so that the compiler emits a shared-memory atomic and a global one (a pointer selected at run time makes
// it a generic-address atomic: measured 213 -> 238 us on the table variant).
__device__ __forceinline__ void scatter9(bool in_table, float* sm, float* gl, V3 b, V3 g) {
    const float bw[3] = {b.x, b.y, b.z};
    if (in_table) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            atomicAdd(sm + 3 * i, bw[i] * g.x);
            atomicAdd(sm + 3 * i + 1, bw[i] * g.y);
            atomicAdd(sm + 3 * i + 2, bw[i] * g.z);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            atomicAdd(gl + 3 * i, bw[i] * g.x);
            atomicAdd(gl + 3 * i + 1, bw[i] * g.y);
            atomicAdd(gl + 3 * i + 2, bw[i] * g.z);
        }
    }
}

// the streaming loop is latency-bound: resident warps matter more than a few spills in the rare branches
// (measured without the cap: 80 -> 120 registers as texel sources were added, 154 -> 224 us)
template <bool TABLE, int NT, bool UV, bool ATLAS>
__global__ void __launch_bounds__(NT, NT <= 128 ? 6 : 1) phong_bwd_kernel(const pert_phong ph, const float* __restrict__ grad_colors,
                                                       float* __restrict__ grad_texels, float* __restrict__ grad_bary,
                                                       float* __restrict__ grad_fv, float* __restrict__ grad_fn, int64_t E,
                                                       int64_t nchunks, int tfaces, int per_image, AtlasSrc at) {
    // dynamic shared memory: [TABLE: F*9 (verts) | F*9 (normals) | F*3 (face colours) or F*9 (corner colours)] then per warp
    // vlist u16[WCHUNK] | hlist u16[WCHUNK] | lighting rows float[2 * PERT_PHONG_STRIDE]
    extern __shared__ __align__(16) float table[];
    constexpr int NWARP = NT / 32;
    constexpr int WARP_BYTES = 2 * WCHUNK * 2 + 2 * PERT_PHONG_STRIDE * 4;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    unsigned char* const wbase = reinterpret_cast<unsigned char*>(table) +
                                 (TABLE ? (((size_t)tfaces * (18 + tex_floats(ph)) * 4 + 15) & ~(size_t)15) : 0) +
                                 (size_t)warp * WARP_BYTES;
    uint16_t* const vlist = reinterpret_cast<uint16_t*>(wbase);
    uint16_t* const hlist = vlist + WCHUNK;
    float* const srow = reinterpret_cast<float*>(hlist + WCHUNK);
    // TABLE: gradients of `tfaces` faces starting at f_begin: the whole mesh, or (per_image) the faces of image
    // blockIdx.y of a batch of equal-size meshes, whose chunks this grid row of CTAs shares; other faces -> global atomics
    const int F = tfaces;
    const int64_t f_begin = (TABLE && per_image) ? (int64_t)blockIdx.y * tfaces : 0;
    float* const t_fv = table;
    float* const t_fn = table + F * 9;
    float* const t_fc = table + F * 18;
    constexpr bool uv_tex = UV;  // UV map: texel gradient scattered into the map (grad_texels = d/d uv_map); its own
                                 // instantiation, so that the common kernels carry none of its code
    // ATLAS: texel gradient added into the atlas cell (grad_texels = d/d atlas), global atomics; its own instantiation too
    const bool face_tex = ATLAS || ph.face_colors || ph.face_vert_colors || uv_tex;  // texel gradient not dense
    const bool vert_tex = ph.face_vert_colors != nullptr;
    const int TF = tex_floats(ph);
    const bool unlit = ph.flags & PERT_PHONG_UNLIT;
    if (TABLE) {
        for (int i = threadIdx.x; i < F * (18 + TF); i += NT) table[i] = 0.0f;
        __syncthreads();
    }
    const bool sparse = ph.flags & PERT_PHONG_SPARSE;
    const int64_t HWK = ph.HW * ph.K;
    int64_t cached_b0 = -1;
    const V3 zero = mk(0.f, 0.f, 0.f);
    const int64_t w0 = (int64_t)blockIdx.x * NWARP + warp, wstride = (int64_t)gridDim.x * NWARP;
    const int64_t e_first = (TABLE && per_image) ? (int64_t)blockIdx.y * HWK : 0;
    const int64_t e_last = (TABLE && per_image) ? e_first + HWK : E;
    const int64_t my_chunks = (TABLE && per_image) ? (HWK + WCHUNK - 1) / WCHUNK : nchunks;
#pragma unroll 1
    for (int64_t c = w0; c < my_chunks; c += wstride) {
        const int64_t e_base = e_first + c * WCHUNK;
        const int Ec = (int)min((int64_t)WCHUNK, e_last - e_base);
        const int vec_ok = ((uintptr_t)(ph.pix_to_face + e_base) & 15) == 0;
        const int64_t b0 = ph.light_rows > 1 ? e_base / HWK : 0;
        if (b0 != cached_b0 && !unlit) {
            __syncwarp();
            fill_rows(ph, b0, srow, lane);
            cached_b0 = b0;
        }
        const RowCache rows{srow, b0, ph.lighting};
        const int64_t* const p2f = ph.pix_to_face + e_base;
        const int nv = scan_valid(p2f, Ec, vec_ok, vlist, WCHUNK);
        __syncwarp();
        if (!sparse && nv < Ec) {
#pragma unroll 1
            for (int i = lane; i < Ec; i += 32) {
                if (__ldg(p2f + i) >= 0) continue;
                const int64_t e = e_base + i;
                if (grad_texels && !face_tex) {
                    const Row L = rows.get(ph.light_rows > 1 ? e / HWK : 0);
                    const V3 gc = ld3(grad_colors + e * 3);
                    st3(grad_texels + e * 3, unlit ? gc : mk(gc.x * L.amb.x, gc.y * L.amb.y, gc.z * L.amb.z));
                }
                if (grad_bary) st3(grad_bary + e * 3, zero);
            }
        }
        // valid entries no sample picked have a zero colour gradient, hence zero gradients everywhere: only the
        // others go on to the lighting arithmetic
        int nh = 0;
#pragma unroll 1
        for (int i0 = 0; i0 < nv; i0 += 32) {
            const int i = i0 + lane;
            bool heavy = false;
            if (i < nv) {
                const int64_t e = e_base + vlist[i];
                const V3 gc = ld3(grad_colors + e * 3);
                heavy = gc.x != 0.0f || gc.y != 0.0f || gc.z != 0.0f;
                if (!heavy) {
                    if (grad_texels && !face_tex) st3(grad_texels + e * 3, zero);
                    if (grad_bary) st3(grad_bary + e * 3, zero);
                }
            }
            const unsigned hb = __ballot_sync(FULL, heavy);
            if (heavy) hlist[nh + __popc(hb & lt)] = vlist[i];
            nh += __popc(hb);
        }
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < nh; i += 32) {
            const int64_t e = e_base + hlist[i];
            const int face = (int)__ldg(ph.pix_to_face + e);
            const int64_t fl = face - f_begin;
            const bool tab = TABLE && fl >= 0 && fl < F;
            const V3 gc = ld3(grad_colors + e * 3);
            const V3 b = ld3(ph.bary + e * 3);
            const V3 t = ATLAS ? atlas_texel(at, face, b) : (UV ? uv_texel(uv_src(ph), e, face, b) : texel_of_plain(ph, e, face, b));
            Row L;
            Lit o;
            V3 v0, v1, v2, n0, n1, n2;
            V3 gt = gc;  // unlit: colour = texel
            if (!unlit) {
                const float* fv = ph.face_verts + (int64_t)face * 9;
                const float* fn = ph.face_normals + (int64_t)face * 9;
                v0 = ld3(fv), v1 = ld3(fv + 3), v2 = ld3(fv + 6);
                n0 = ld3(fn), n1 = ld3(fn + 3), n2 = ld3(fn + 6);
                L = rows.get(ph.light_rows > 1 ? e / HWK : 0);
                o = light_entry(L, b.x * v0 + b.y * v1 + b.z * v2, b.x * n0 + b.y * n1 + b.z * n2);
                // colour = (amb + dif * ang) * t + spc * pw
                gt = mk(gc.x * (L.amb.x + L.dif.x * o.ang), gc.y * (L.amb.y + L.dif.y * o.ang), gc.z * (L.amb.z + L.dif.z * o.ang));
            }
            V3 gb = zero;  // gradient of bary_coords
            if (vert_tex) gb = vert_texel_bary_grad(ph.face_vert_colors + (int64_t)face * 9, gt);  // texel = sum_i b_i C_i
            if (uv_tex) {  // texel = bilinear(map, sum_i b_i uv_i): gradient to the four taps and, through (u, v), to bary
                gb = uv_texel_bwd(uv_src(ph), e, face, b, gt, grad_texels);
            } else if (ATLAS) {  // texel = atlas[face, cell(b)]: piecewise constant in b, nothing to bary
                if (grad_texels) {
                    float* dst = grad_texels + atlas_cell(at, face, b.x, b.y);
                    atomicAdd(dst, gt.x);
                    atomicAdd(dst + 1, gt.y);
                    atomicAdd(dst + 2, gt.z);
                }
            } else if (grad_texels) {
                if (vert_tex) {
                    scatter9(tab, t_fc + fl * 9, grad_texels + (int64_t)face * 9, b, gt);
                } else if (face_tex) {
                    if (tab) {  // separate statements: a shared-memory atomic and a global one, not a generic one
                        atomicAdd(t_fc + fl * 3, gt.x);
                        atomicAdd(t_fc + fl * 3 + 1, gt.y);
                        atomicAdd(t_fc + fl * 3 + 2, gt.z);
                    } else {
                        float* dst = grad_texels + (int64_t)face * 3;
                        atomicAdd(dst, gt.x);
                        atomicAdd(dst + 1, gt.y);
                        atomicAdd(dst + 2, gt.z);
                    }
                } else {
                    st3(grad_texels + e * 3, gt);
                }
            }
            if (unlit) {
                if (grad_bary) st3(grad_bary + e * 3, gb);
                continue;
            }
            const float g_ang = gc.x * L.dif.x * t.x + gc.y * L.dif.y * t.y + gc.z * L.dif.z * t.z;
            const float g_pw = gc.x * L.spc.x + gc.y * L.spc.y + gc.z * L.spc.z;
            // pw = alpha^sh; alpha = relu(v.r) * [n.d > 0]   (torch's pow backward: 0 at alpha = 0)
            const float g_vr = (o.alpha > 0.0f && L.sh != 0.0f) ? g_pw * L.sh * powf(o.alpha, L.sh - 1.0f) : 0.0f;
            const V3 g_v = g_vr * o.r, g_r = g_vr * o.v;
            // r = 2 cos n - d; ang = relu(cos); cos = n.d
            const float g_cos = 2.0f * dot(g_r, o.n) + (o.cosd > 0.0f ? g_ang : 0.0f);
            const V3 g_n = (2.0f * o.cosd) * g_r + g_cos * o.d;
            const V3 g_d = g_cos * o.n - g_r;
            const V3 g_nraw = normalize_bwd(o.n, o.nl, g_n);
            const V3 g_vraw = normalize_bwd(o.v, o.vl, g_v);
            V3 g_p = mk(-g_vraw.x, -g_vraw.y, -g_vraw.z);
            if (!L.directional) g_p = g_p - normalize_bwd(o.d, o.dl, g_d);
            if (grad_bary)
                st3(grad_bary + e * 3, mk(gb.x + dot(g_p, v0) + dot(g_nraw, n0), gb.y + dot(g_p, v1) + dot(g_nraw, n1),
                                          gb.z + dot(g_p, v2) + dot(g_nraw, n2)));
            if (grad_fv) scatter9(tab, t_fv + fl * 9, grad_fv + (int64_t)face * 9, b, g_p);
            if (grad_fn) scatter9(tab, t_fn + fl * 9, grad_fn + (int64_t)face * 9, b, g_nraw);
        }
        __syncwarp();
    }
    if (TABLE) {
        __syncthreads();
        for (int i = threadIdx.x; i < F * 9; i += NT) {
            if (grad_fv && t_fv[i] != 0.0f) atomicAdd(grad_fv + f_begin * 9 + i, t_fv[i]);
            if (grad_fn && t_fn[i] != 0.0f) atomicAdd(grad_fn + f_begin * 9 + i, t_fn[i]);
        }
        if (face_tex && !uv_tex && grad_texels)
            for (int i = threadIdx.x; i < F * TF; i += NT)
                if (t_fc[i] != 0.0f) atomicAdd(grad_texels + f_begin * TF + i, t_fc[i]);
    }
}


// Gradient of the lighting table (light location / direction, the three material x light colour products, shininess,
// camera centre): a second sparse pass launched only when the caller asks for it (lights and cameras are constants in
// the reference's pose optimisation, eval.py:233-262, but eval.py:411-470 and :693-725 optimise them).  Every lane
// keeps the sixteen sums of its entries in registers and adds them to grad_lighting once (per row of the table).
template <bool ATLAS>
__global__ void __launch_bounds__(PT) phong_light_bwd_kernel(const pert_phong ph, const float* __restrict__ grad_colors,
                                                             float* __restrict__ grad_lighting, int64_t E, int64_t nchunks,
                                                             AtlasSrc at) {
    __shared__ __align__(16) uint16_t s_vlist[PW][WCHUNK];
    __shared__ float s_row[PW][2 * PERT_PHONG_STRIDE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t* const vlist = s_vlist[warp];
    float* const srow = s_row[warp];
    const int64_t HWK = ph.HW * ph.K;
    int64_t cached_b0 = -1, acc_row = -1;
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.0f;
    auto flush = [&]() {
        if (acc_row < 0) return;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            if (acc[i] != 0.0f) atomicAdd(grad_lighting + acc_row * PERT_PHONG_STRIDE + i, acc[i]);
            acc[i] = 0.0f;
        }
    };
    const int64_t w0 = (int64_t)blockIdx.x * PW + warp, wstride = (int64_t)gridDim.x * PW;
#pragma unroll 1
    for (int64_t c = w0; c < nchunks; c += wstride) {
        const int64_t e_base = c * WCHUNK;
        const int Ec = (int)min((int64_t)WCHUNK, E - e_base);
        const int vec_ok = ((uintptr_t)(ph.pix_to_face + e_base) & 15) == 0;
        const int64_t b0 = ph.light_rows > 1 ? e_base / HWK : 0;
        if (b0 != cached_b0) {
            __syncwarp();
            fill_rows(ph, b0, srow, lane);
            cached_b0 = b0;
        }
        const RowCache rows{srow, b0, ph.lighting};
        const int nv = scan_valid(ph.pix_to_face + e_base, Ec, vec_ok, vlist, WCHUNK);
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < nv; i += 32) {
            const int64_t e = e_base + vlist[i];
            const V3 gc = ld3(grad_colors + e * 3);
            if (gc.x == 0.0f && gc.y == 0.0f && gc.z == 0.0f) continue;
            const int64_t face = __ldg(ph.pix_to_face + e);
            const V3 b = ld3(ph.bary + e * 3);
            const V3 t = texel_src<ATLAS>(ph, at, e, face, b);
            const float* fv = ph.face_verts + face * 9;
            const float* fn = ph.face_normals + face * 9;
            const V3 p = b.x * ld3(fv) + b.y * ld3(fv + 3) + b.z * ld3(fv + 6);
            const V3 nr = b.x * ld3(fn) + b.y * ld3(fn + 3) + b.z * ld3(fn + 6);
            const int64_t row = ph.light_rows > 1 ? e / HWK : 0;
            const Row L = rows.get(row);
            const Lit o = light_entry(L, p, nr);
            if (row != acc_row) {
                flush();
                acc_row = row;
            }
            // colour = (amb + dif * ang) * t + spc * pw
            const float g_ang = gc.x * L.dif.x * t.x + gc.y * L.dif.y * t.y + gc.z * L.dif.z * t.z;
            const float g_pw = gc.x * L.spc.x + gc.y * L.spc.y + gc.z * L.spc.z;
            const float g_vr = (o.alpha > 0.0f && L.sh != 0.0f) ? g_pw * L.sh * powf(o.alpha, L.sh - 1.0f) : 0.0f;
            const V3 g_v = g_vr * o.r, g_r = g_vr * o.v;
            const float g_cos = 2.0f * dot(g_r, o.n) + (o.cosd > 0.0f ? g_ang : 0.0f);
            const V3 g_d = g_cos * o.n - g_r;
            const V3 g_loc = normalize_bwd(o.d, o.dl, g_d);   // d_raw = loc - p (point) or loc (directional)
            const V3 g_cam = normalize_bwd(o.v, o.vl, g_v);   // v_raw = cam - p
            acc[0] += g_loc.x, acc[1] += g_loc.y, acc[2] += g_loc.z;
            acc[3] += gc.x * t.x, acc[4] += gc.y * t.y, acc[5] += gc.z * t.z;
            acc[6] += gc.x * t.x * o.ang, acc[7] += gc.y * t.y * o.ang, acc[8] += gc.z * t.z * o.ang;
            acc[9] += gc.x * o.pw, acc[10] += gc.y * o.pw, acc[11] += gc.z * o.pw;
            if (o.alpha > 0.0f) acc[12] += g_pw * o.pw * logf(o.alpha);  // d alpha^sh / d sh
            acc[13] += g_cam.x, acc[14] += g_cam.y, acc[15] += g_cam.z;
        }
        __syncwarp();
    }
    // one add per warp when all its lanes hold sums of the same row (the usual case), else one per lane
    const int64_t rr = (int64_t)warp_max_i((int)acc_row);  // rows fit 32 bits
    const bool uniform = __all_sync(FULL, acc_row == rr || acc_row < 0);
    if (uniform) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const float v = warp_sum(acc_row >= 0 ? acc[i] : 0.0f);
            if (lane == 0 && rr >= 0 && v != 0.0f) atomicAdd(grad_lighting + rr * PERT_PHONG_STRIDE + i, v);
        }
    } else {
        flush();
    }
}

unsigned phong_grid(int64_t nchunks, int ctas_per_sm, int warps_per_cta = PW) {
    const int64_t cap = sm_count() * (int64_t)ctas_per_sm, need = (nchunks + warps_per_cta - 1) / warps_per_cta;
    return (unsigned)(need < cap ? need : cap);
}

}  // namespace

static int vec_ok_of(const pert_phong& ph) { return ((uintptr_t)ph.pix_to_face & 15) == 0; }

int launch_phong_fwd(const pert_phong& ph, float* colors, cudaStream_t st, const float* atlas, int atlas_r) {
    const int64_t E = ph.P * ph.K, nchunks = (E + WCHUNK - 1) / WCHUNK;
    const AtlasSrc at{atlas, atlas_r};
    if (atlas)
        phong_fwd_kernel<true><<<phong_grid(nchunks, 9), PT, 0, st>>>(ph, colors, E, nchunks, vec_ok_of(ph), at);
    else
        phong_fwd_kernel<false><<<phong_grid(nchunks, 9), PT, 0, st>>>(ph, colors, E, nchunks, vec_ok_of(ph), at);
    return (int)cudaGetLastError();
}

template <bool TABLE, int NT, bool UV = false, bool ATLAS = false>
static int launch_bwd_t(const pert_phong& ph, const float* grad_colors, float* grad_texels, float* grad_bary, float* grad_fv,
                        float* grad_fn, int64_t E, int64_t nchunks, int ctas_per_sm, int tfaces, bool per_image, cudaStream_t st,
                        AtlasSrc at = AtlasSrc{nullptr, 0}) {
    const size_t table = TABLE ? (((size_t)tfaces * (18 + tex_floats(ph)) * 4 + 15) & ~(size_t)15) : 0;
    const size_t smem = table + (size_t)(NT / 32) * (2 * WCHUNK * 2 + 2 * PERT_PHONG_STRIDE * 4);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(phong_bwd_kernel<TABLE, NT, UV, ATLAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    dim3 grid(phong_grid(nchunks, ctas_per_sm, NT / 32));
    if (per_image) {  // one grid row of CTAs per image, about one CTA per SM in total
        const int64_t n_img = ph.P / ph.HW, img_chunks = (ph.HW * ph.K + WCHUNK - 1) / WCHUNK;
        int64_t ctas = (sm_count() * (int64_t)ctas_per_sm + n_img - 1) / n_img;
        const int64_t most = (img_chunks + NT / 32 - 1) / (NT / 32);
        grid = dim3((unsigned)(ctas < most ? ctas : most), (unsigned)n_img);
    }
    phong_bwd_kernel<TABLE, NT, UV, ATLAS><<<grid, NT, smem, st>>>(ph, grad_colors, grad_texels, grad_bary, grad_fv, grad_fn, E,
                                                                  nchunks, tfaces, per_image ? 1 : 0, at);
    return (int)cudaGetLastError();
}

int launch_phong_light_bwd(const pert_phong& ph, const float* grad_colors, float* grad_lighting, cudaStream_t st,
                           const float* atlas, int atlas_r) {
    const int64_t E = ph.P * ph.K, nchunks = (E + WCHUNK - 1) / WCHUNK;
    const AtlasSrc at{atlas, atlas_r};
    if (atlas)
        phong_light_bwd_kernel<true><<<phong_grid(nchunks, 4), PT, 0, st>>>(ph, grad_colors, grad_lighting, E, nchunks, at);
    else
        phong_light_bwd_kernel<false><<<phong_grid(nchunks, 4), PT, 0, st>>>(ph, grad_colors, grad_lighting, E, nchunks, at);
    return (int)cudaGetLastError();
}

int launch_phong_bwd(const pert_phong& ph, const float* grad_colors, float* grad_texels, float* grad_bary, float* grad_fv,
                     float* grad_fn, cudaStream_t st, const float* atlas, int atlas_r) {
    const int64_t E = ph.P * ph.K, nchunks = (E + WCHUNK - 1) / WCHUNK;
    // Atlas: its own instantiation, every gradient straight to global memory.  A ShapeNet atlas (tens of thousands of
    // faces) is far beyond the shared-memory table, and so are the face-vertex and normal tables of such a mesh
    if (atlas)
        return launch_bwd_t<false, PT, false, true>(ph, grad_colors, grad_texels, grad_bary, grad_fv, grad_fn, E, nchunks, 6, 0,
                                                    false, st, AtlasSrc{atlas, atlas_r});
    const bool scatter = grad_fv || grad_fn || (tex_floats(ph) && grad_texels);
    const size_t per_face = (size_t)(18 + tex_floats(ph)) * 4;
    // Small meshes: every entry's 18 atomic adds would land on the same few thousand L2 addresses (measured at
    // 1280 faces: 210 us of a 360 us pass); accumulate them in a per-SM shared-memory table instead and flush it
    // once.  Large meshes spread the atomics over enough addresses (100k faces: 58 us).  A batch of N equal-size
    // meshes (N poses of one topology: faces_per_mesh) gets one table per image.
    if (ph.uv_map)  // rare path: its own instantiation, face-table gradients straight to global memory
        return launch_bwd_t<false, PT, true>(ph, grad_colors, grad_texels, grad_bary, grad_fv, grad_fn, E, nchunks, 6, 0, false, st);
    const int64_t n_img = ph.P / ph.HW;
    // per-image tables only for small meshes: measured on a batch of 8 x 1280 faces with real (dense) fragments, the
    // shared-memory CAS adds of the one-CTA-per-SM table kernel (683 us) lose to plain L2 reductions spread over
    // 8 x 23 k addresses (427 us); contention on L2 is the problem of SMALL tables only
    const bool batch = ph.faces_per_mesh > 0 && ph.faces_per_mesh <= 256 && n_img > 1 && ph.faces_per_mesh * n_img == ph.num_faces &&
                       n_img <= 65535 && ph.HW * ph.K >= 4 * (int64_t)(PT_TABLE / 32) * WCHUNK;
    const int64_t tf = batch ? ph.faces_per_mesh : ph.num_faces;
    if (scatter && tf * per_face <= 16 * 1024 && !batch)  // tiny table: keep the occupancy of the small CTAs
        return launch_bwd_t<true, PT>(ph, grad_colors, grad_texels, grad_bary, grad_fv, grad_fn, E, nchunks, 4, (int)tf, false, st);
    if (scatter && tf * per_face <= (size_t)TABLE_MAX_BYTES)
        return launch_bwd_t<true, PT_TABLE>(ph, grad_colors, grad_texels, grad_bary, grad_fv, grad_fn, E, nchunks, 1, (int)tf, batch, st);
    return launch_bwd_t<false, PT>(ph, grad_colors, grad_texels, grad_bary, grad_fv, grad_fn, E, nchunks, 6, 0, false, st);
}

}  // namespace pert
