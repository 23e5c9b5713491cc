// Texel lookups shared by the Phong kernels (phong.cu) and the fused shading kernels (shade_fwd.cu, shade_bwd.cu): vertex
// colours interpolated with the barycentric coordinates, bilinear UV taps and atlas cells.  Both sides call these
// functions, so that a texel sampled inside the fused kernels is the same float expression as the one the texture-only
// Phong kernel (PERT_PHONG_UNLIT) materialises.
#pragma once
#include "kernels.h"

namespace pert {

namespace {

struct V3 {
    float x, y, z;
};
__device__ __forceinline__ V3 mk(float x, float y, float z) { return V3{x, y, z}; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ V3 operator*(float s, V3 a) { return mk(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 ld3(const float* p) { return mk(__ldg(p), __ldg(p + 1), __ldg(p + 2)); }
__device__ __forceinline__ void st3(float* p, V3 v) {
    p[0] = v.x;
    p[1] = v.y;
    p[2] = v.z;
}

// Colours at the three corners of a face, c = (3,3) row of the (F,3,3) table, interpolated with bary (TexturesVertex)
__device__ __forceinline__ V3 vert_texel(const float* c, V3 b) { return b.x * ld3(c) + b.y * ld3(c + 3) + b.z * ld3(c + 6); }
// its gradient with respect to bary for a texel gradient gt: <C_i, gt>
__device__ __forceinline__ V3 vert_texel_bary_grad(const float* c, V3 gt) { return mk(dot(gt, ld3(c)), dot(gt, ld3(c + 3)), dot(gt, ld3(c + 6))); }

// Bilinear tap of a UV map, torch.nn.functional.grid_sample(mode="bilinear", padding_mode="border",
// align_corners=True) on the vertically flipped map, as pytorch3d 0.4.0's TexturesUV.sample_textures does:
// column = u (Wm-1), row = (Hm-1) - v (Hm-1), both clamped to the map.
// The UV path is rare: it lives in out-of-line functions that take this small record BY VALUE (a reference to the
// kernel's parameter struct would force a local-memory copy of it in every kernel: measured +60 % on backward).
struct UvSrc {
    const float* uv_map;
    const float* face_uvs;
    int map_h, map_w, map_count;
    int64_t HWK;
};
__device__ __forceinline__ UvSrc uv_src(const pert_phong& ph) {
    return UvSrc{ph.uv_map, ph.face_uvs, ph.map_h, ph.map_w, ph.map_count, ph.HW * ph.K};
}
struct UvTap {
    int x0, y0, x1, y1;
    float fx, fy;   // fractional parts
    bool cx, cy;    // coordinate clamped by the border rule: its gradient is zero
};
__device__ __forceinline__ UvTap uv_tap(const UvSrc& us, float u, float v) {
    const float wm = (float)(us.map_w - 1), hm = (float)(us.map_h - 1);
    float ix = u * wm, iy = hm - v * hm;
    UvTap t;
    t.cx = !(ix > 0.0f && ix < wm);
    t.cy = !(iy > 0.0f && iy < hm);
    ix = fminf(fmaxf(ix, 0.0f), wm);
    iy = fminf(fmaxf(iy, 0.0f), hm);
    const float fx0 = floorf(ix), fy0 = floorf(iy);
    t.x0 = (int)fx0;
    t.y0 = (int)fy0;
    t.x1 = min(t.x0 + 1, us.map_w - 1);
    t.y1 = min(t.y0 + 1, us.map_h - 1);
    t.fx = ix - fx0;
    t.fy = iy - fy0;
    return t;
}
__device__ __forceinline__ int64_t uv_map_offset(const UvSrc& us, int64_t e) {
    return (us.map_count > 1 ? e / us.HWK : 0) * (int64_t)us.map_h * us.map_w * 3;
}

__device__ __noinline__ V3 uv_texel(UvSrc us, int64_t e, int64_t face, V3 b) {
    const float* q = us.face_uvs + face * 6;
    const float u = b.x * __ldg(q) + b.y * __ldg(q + 2) + b.z * __ldg(q + 4);
    const float v = b.x * __ldg(q + 1) + b.y * __ldg(q + 3) + b.z * __ldg(q + 5);
    const UvTap t = uv_tap(us, u, v);
    const float* m = us.uv_map + uv_map_offset(us, e);
    const V3 c00 = ld3(m + ((int64_t)t.y0 * us.map_w + t.x0) * 3), c01 = ld3(m + ((int64_t)t.y0 * us.map_w + t.x1) * 3);
    const V3 c10 = ld3(m + ((int64_t)t.y1 * us.map_w + t.x0) * 3), c11 = ld3(m + ((int64_t)t.y1 * us.map_w + t.x1) * 3);
    const float w00 = (1.0f - t.fx) * (1.0f - t.fy), w01 = t.fx * (1.0f - t.fy), w10 = (1.0f - t.fx) * t.fy, w11 = t.fx * t.fy;
    return w00 * c00 + w01 * c01 + w10 * c10 + w11 * c11;
}
// gradient of the UV texel: adds w_tap * gt to the four taps of grad_map (may be NULL), returns d/d bary
__device__ __noinline__ V3 uv_texel_bwd(UvSrc us, int64_t e, int64_t face, V3 b, V3 gt, float* grad_map) {
    const float* q = us.face_uvs + face * 6;
    const float u = b.x * __ldg(q) + b.y * __ldg(q + 2) + b.z * __ldg(q + 4);
    const float v = b.x * __ldg(q + 1) + b.y * __ldg(q + 3) + b.z * __ldg(q + 5);
    const UvTap tp = uv_tap(us, u, v);
    const int64_t mo = uv_map_offset(us, e);
    const float* m = us.uv_map + mo;
    const int64_t i00 = ((int64_t)tp.y0 * us.map_w + tp.x0) * 3, i01 = ((int64_t)tp.y0 * us.map_w + tp.x1) * 3;
    const int64_t i10 = ((int64_t)tp.y1 * us.map_w + tp.x0) * 3, i11 = ((int64_t)tp.y1 * us.map_w + tp.x1) * 3;
    const V3 c00 = ld3(m + i00), c01 = ld3(m + i01), c10 = ld3(m + i10), c11 = ld3(m + i11);
    // d texel / d column, d texel / d row
    const V3 dx = (1.0f - tp.fy) * (c01 - c00) + tp.fy * (c11 - c10);
    const V3 dy = (1.0f - tp.fx) * (c10 - c00) + tp.fx * (c11 - c01);
    const float g_u = tp.cx ? 0.0f : dot(gt, dx) * (float)(us.map_w - 1);
    const float g_v = tp.cy ? 0.0f : -dot(gt, dy) * (float)(us.map_h - 1);
    if (grad_map) {
        float* gm = grad_map + mo;
        const float w[4] = {(1.0f - tp.fx) * (1.0f - tp.fy), tp.fx * (1.0f - tp.fy), (1.0f - tp.fx) * tp.fy, tp.fx * tp.fy};
        const int64_t idx[4] = {i00, i01, i10, i11};
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
            atomicAdd(gm + idx[k4], w[k4] * gt.x);
            atomicAdd(gm + idx[k4] + 1, w[k4] * gt.y);
            atomicAdd(gm + idx[k4] + 2, w[k4] * gt.z);
        }
    }
    return mk(g_u * __ldg(q) + g_v * __ldg(q + 1), g_u * __ldg(q + 2) + g_v * __ldg(q + 3), g_u * __ldg(q + 4) + g_v * __ldg(q + 5));
}

// Per-face texture atlas (TexturesAtlas; the ShapeNet models of experiments/eval.py:216-238): atlas (F,R,R,3), an R x R
// grid of texels per packed face.  pert_phong has no room for it, so the atlas kernels take this record as a parameter of
// their own, BY VALUE for the reason given at UvSrc; only the ATLAS instantiations read it.
struct AtlasSrc {
    const float* atlas;
    int R;
};
// Float offset of the cell that (w0, w1) picks: AtlasTexels.materialize's rule (structures.py), op for op in float32 --
// torch.nan_to_num (NaN -> 0, +-inf -> +-FLT_MAX); w R rounded once, clamped to [-1, R] before the truncation, then to
// R - 1; the point is below the diagonal when (w0 + w1) R - (wx + wy) <= 1 (each op rounded once, no FMA), else the cell
// is reflected; finally clamped to the grid.
// The barycentric coordinates of the rasteriser are unclipped (outside [0, 1] in the blur band): every cell stays in range.
// num_faces R^2 3 < 2^31 (pert_phong_atlas_fwd refuses larger atlases): 32-bit offsets.
__device__ __forceinline__ int atlas_cell(AtlasSrc a, int face, float w0, float w1) {
    const float rf = (float)a.R;
    w0 = isnan(w0) ? 0.0f : fminf(fmaxf(w0, -CUDART_MAX_NORMAL_F), CUDART_MAX_NORMAL_F);
    w1 = isnan(w1) ? 0.0f : fminf(fmaxf(w1, -CUDART_MAX_NORMAL_F), CUDART_MAX_NORMAL_F);
    int wx = min((int)fminf(fmaxf(__fmul_rn(w0, rf), -1.0f), rf), a.R - 1);
    int wy = min((int)fminf(fmaxf(__fmul_rn(w1, rf), -1.0f), rf), a.R - 1);
    if (!(__fsub_rn(__fmul_rn(__fadd_rn(w0, w1), rf), (float)(wx + wy)) <= 1.0f)) {
        wx = a.R - 1 - wx;
        wy = a.R - 1 - wy;
    }
    wx = min(max(wx, 0), a.R - 1);
    wy = min(max(wy, 0), a.R - 1);
    return ((face * a.R + wy) * a.R + wx) * 3;
}
__device__ __forceinline__ V3 atlas_texel(AtlasSrc a, int64_t face, V3 b) { return ld3(a.atlas + atlas_cell(a, (int)face, b.x, b.y)); }

// Texel of entry e (index into the (P,K) entries of the call) of face `face` with barycentric coordinates b, from a
// pert_texture source (TEX = TX_VERT, TX_UV or TX_ATLAS): the fused kernels' counterpart of phong.cu's texel_src.  HWK =
// entries per image (selects the UV map when there is one per image)
template <int TEX>
__device__ __forceinline__ V3 tex_texel(const TexArgs& t, int64_t HWK, int64_t e, int64_t face, V3 b) {
    if constexpr (TEX == TX_VERT) return vert_texel(t.table + face * 9, b);
    else if constexpr (TEX == TX_UV) return uv_texel(UvSrc{t.table, t.face_uvs, t.map_h, t.map_w, t.map_count, HWK}, e, face, b);
    else return atlas_texel(AtlasSrc{t.table, t.R}, face, b);
}
// Backward of tex_texel for the texel gradient g: atomic adds into grad_table (may be NULL), as pert_phong_bwd scatters
// them (vertex colours: b_i g into corner i; UV: the four taps; atlas: the cell); returns the gradient of b (0 for the
// atlas, whose texel is piecewise constant in b)
template <int TEX>
__device__ __forceinline__ V3 tex_texel_bwd(const TexArgs& t, int64_t HWK, int64_t e, int64_t face, V3 b, V3 g, float* grad_table) {
    if constexpr (TEX == TX_VERT) {
        if (grad_table) {
            float* dst = grad_table + face * 9;
            const float bw[3] = {b.x, b.y, b.z};
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                atomicAdd(dst + 3 * i, bw[i] * g.x);
                atomicAdd(dst + 3 * i + 1, bw[i] * g.y);
                atomicAdd(dst + 3 * i + 2, bw[i] * g.z);
            }
        }
        return vert_texel_bary_grad(t.table + face * 9, g);
    } else if constexpr (TEX == TX_UV) {
        return uv_texel_bwd(UvSrc{t.table, t.face_uvs, t.map_h, t.map_w, t.map_count, HWK}, e, face, b, g, grad_table);
    } else {
        if (grad_table) {
            float* dst = grad_table + atlas_cell(AtlasSrc{t.table, t.R}, (int)face, b.x, b.y);
            atomicAdd(dst, g.x);
            atomicAdd(dst + 1, g.y);
            atomicAdd(dst + 2, g.z);
        }
        return mk(0.f, 0.f, 0.f);
    }
}

}  // namespace

}  // namespace pert
