// Fragment producer (pert_rasterize_fwd / pert_rasterize_bwd in include/pertshade.h): the K-deep Fragments
// (pix_to_face, zbuf, bary_coords, dists) the perturbed shader consumes.  The reference gets them from pytorch3d's
// MeshRasterizer (experiments/eval.py:135-141,165-169: blur_radius = log(1/1e-4 - 1) * sigma, faces_per_pixel = 50,
// perspective_correct = False); pytorch3d 0.4.0 (requirements.txt:7) is not under the reference tree, so this
// restates its published naive rasteriser (rasterize_meshes.cu CheckPixelInsideFace / RasterizeMeshesNaive,
// geometry_utils.cuh, kEpsilon = 1e-8) with a B200 work decomposition:
//
//   forward   one CTA per 32x4 pixel tile.  Faces are culled against the tile in chunks of 256 (one face per thread:
//             bounding box grown by sqrt(blur_radius) against the tile's pixel-centre rectangle, zero-area and
//             behind-camera faces dropped), survivors are compacted IN FACE ORDER into shared memory with their nine
//             coordinates, and every pixel thread then tests only those.  The K-buffer of a pixel is a sorted array
//             of packed keys (depth bits << 32 | face) in local memory for K <= 64, or lives in the pixel's own
//             output rows for larger K (stable insertion: ascending depth, ties in face order); bary / dists of the
//             kept faces are recomputed at the end and the padding of each row is written by the warp as coalesced
//             stores.
//   bins      for large meshes (K <= 64), candidate lists per tile built by one thread per face in two passes (count,
//             then fill) around the caller's prefix sum.  pert_rasterize_bin lists a face in every tile its box
//             overlaps, so the total length is only known on the device.  pert_rasterize_bin_bounded lists a face in
//             at most RASTER_BIN_CAP tiles and puts a face that overlaps more into one wide list per image, which every
//             tile of the image walks after its own: the total is at most RASTER_BIN_CAP * num_faces, the caller sizes
//             the lists from shapes alone, and the render needs no host synchronisation (CUDA-graph capturable).
//   backward  a streaming pass over the (P,K) entries, warp-autonomous chunks with compact valid lists (the machinery
//             of the Phong kernels): every valid entry recomputes its barycentric / distance arithmetic and scatters
//             d(zbuf, bary, dists)/d(face_verts) with atomics.
#include "kernels.h"
#include "tile.cuh"

namespace pert {

namespace {

constexpr float kEps = 1e-8f;  // geometry_utils.cuh kEpsilon
constexpr int TW = 32, TH = 4, RT = TW * TH;  // pixel tile of the forward kernel (K = 50: 50 KB of K-buffers, 3 CTAs per SM)

struct P2 {
    float x, y;
};
__device__ __forceinline__ P2 operator-(P2 a, P2 b) { return P2{a.x - b.x, a.y - b.y}; }
__device__ __forceinline__ float dot2(P2 a, P2 b) { return a.x * b.x + a.y * b.y; }

// rasterize_meshes.cu PixToNonSquareNdc: centre of pixel i along an axis of S1 pixels (other axis S2)
__device__ __forceinline__ float pix_to_ndc(int i, int S1, int S2) {
    const float range = S1 > S2 ? (float)S1 / (float)S2 : 1.0f;
    return -range + (2.0f * (float)i + 1.0f) * range / (float)S1;
}

// geometry_utils.cuh EdgeFunctionForward
__device__ __forceinline__ float edge(P2 p, P2 a, P2 b) { return (p.x - a.x) * (b.y - a.y) - (p.y - a.y) * (b.x - a.x); }

// geometry_utils.cuh PointLineDistanceForward: squared distance to the segment a-b; tt = clamped parameter
__device__ __forceinline__ float point_line(P2 p, P2 a, P2 b, float& tt, bool& degenerate) {
    const P2 ab = b - a;
    const float l2 = dot2(ab, ab);
    degenerate = l2 <= kEps;
    if (degenerate) {
        tt = 1.0f;
        return dot2(p - b, p - b);
    }
    const float t = dot2(ab, p - a) / l2;
    tt = fminf(fmaxf(t, 0.0f), 1.0f);
    const P2 r = p - P2{a.x + tt * ab.x, a.y + tt * ab.y};
    return dot2(r, r);
}

struct FaceEval {
    float w0, w1, w2, area, pz, dist;
    int min_edge;  // 0: v0-v1, 1: v0-v2, 2: v1-v2
    bool inside;
};

// bary (unclipped, not perspective-corrected), interpolated depth, squared distance to the triangle
__device__ __forceinline__ FaceEval eval_face(P2 p, const float* v /* 9 floats */) {
    const P2 v0{v[0], v[1]}, v1{v[3], v[4]}, v2{v[6], v[7]};
    FaceEval o;
    o.area = edge(v2, v0, v1) + kEps;  // BarycentricCoordsForward
    o.w0 = edge(p, v1, v2) / o.area;
    o.w1 = edge(p, v2, v0) / o.area;
    o.w2 = edge(p, v0, v1) / o.area;
    o.pz = o.w0 * v[2] + o.w1 * v[5] + o.w2 * v[8];
    float tt;
    bool dg;
    const float e01 = point_line(p, v0, v1, tt, dg), e02 = point_line(p, v0, v2, tt, dg), e12 = point_line(p, v1, v2, tt, dg);
    o.dist = e01;
    o.min_edge = 0;
    if (e02 < o.dist) {
        o.dist = e02;
        o.min_edge = 1;
    }
    if (e12 < o.dist) {
        o.dist = e12;
        o.min_edge = 2;
    }
    o.inside = o.w0 > 0.0f && o.w1 > 0.0f && o.w2 > 0.0f;
    return o;
}

// ---------------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RT) rasterize_fwd_rows_kernel(const pert_raster rs, int64_t* __restrict__ pix_to_face,
                                                           float* __restrict__ zbuf, float* __restrict__ bary,
                                                           float* __restrict__ dists) {
    __shared__ float s_v[RT][9];
    __shared__ int s_face[RT];
    __shared__ int s_wcount[RT / 32];
    const int H = rs.H, W = rs.W, K = rs.K;
    const int n = blockIdx.z, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int px = blockIdx.x * TW + lane, py = blockIdx.y * TH + warp;  // column / row of this thread's pixel
    const bool in_image = px < W && py < H;
    // pixel (0,0) is the top-left corner; NDC has +X left and +Y up (RasterizeMeshesNaiveCudaKernel)
    const P2 p{pix_to_ndc(W - 1 - px, W, H), pix_to_ndc(H - 1 - py, H, W)};
    // pixel-centre rectangle of the tile (clipped to the image)
    const int px0 = blockIdx.x * TW, px1 = min(px0 + TW, W) - 1, py0 = blockIdx.y * TH, py1 = min(py0 + TH, H) - 1;
    const float tx_hi = pix_to_ndc(W - 1 - px0, W, H), tx_lo = pix_to_ndc(W - 1 - px1, W, H);
    const float ty_hi = pix_to_ndc(H - 1 - py0, H, W), ty_lo = pix_to_ndc(H - 1 - py1, H, W);
    const float blur = rs.blur_radius, r = sqrtf(blur);
    const int64_t f_begin = __ldg(rs.face_start + n), f_end = __ldg(rs.face_start + n + 1);
    const int64_t row = (((int64_t)n * H + py) * W + px) * K;  // this pixel's K-buffer = its output rows
    int cnt = 0;

#pragma unroll 1
    for (int64_t fc = f_begin; fc < f_end; fc += RT) {
        // ---- cull one face per thread against the tile --------------------------------------------------
        const int64_t f = fc + threadIdx.x;
        bool keep = false;
        float v[9];
        if (f < f_end) {
#pragma unroll
            for (int i = 0; i < 9; ++i) v[i] = __ldg(rs.face_verts + f * 9 + i);
            const float xmin = fminf(fminf(v[0], v[3]), v[6]) - r, xmax = fmaxf(fmaxf(v[0], v[3]), v[6]) + r;
            const float ymin = fminf(fminf(v[1], v[4]), v[7]) - r, ymax = fmaxf(fmaxf(v[1], v[4]), v[7]) + r;
            const float zmax = fmaxf(fmaxf(v[2], v[5]), v[8]);
            const float area = edge(P2{v[0], v[1]}, P2{v[3], v[4]}, P2{v[6], v[7]});
            const bool zero_area = area <= kEps && area >= -kEps;
            const bool back = (rs.flags & PERT_RAST_CULL_BACKFACES) && area < 0.0f;
            keep = !(zmax < 0.0f) && !zero_area && !back && !(tx_lo > xmax || tx_hi < xmin || ty_lo > ymax || ty_hi < ymin);
        }
        const unsigned b = __ballot_sync(FULL, keep);
        if (lane == 0) s_wcount[warp] = __popc(b);
        __syncthreads();  // also: the previous chunk's list has been consumed
        int base = 0, total = 0;
#pragma unroll
        for (int w = 0; w < RT / 32; ++w) {
            const int c = s_wcount[w];
            base += w < warp ? c : 0;
            total += c;
        }
        if (keep) {  // ordered compaction: faces stay in index order (depth ties are resolved by face order)
            const int pos = base + __popc(b & ((1u << lane) - 1u));
            s_face[pos] = (int)(f - f_begin);
#pragma unroll
            for (int i = 0; i < 9; ++i) s_v[pos][i] = v[i];
        }
        __syncthreads();
        // ---- every pixel tests the surviving faces (CheckPixelInsideFace) ---------------------------------
        if (in_image) {
#pragma unroll 1
            for (int i = 0; i < total; ++i) {
                const float* fv = s_v[i];
                const float xmin = fminf(fminf(fv[0], fv[3]), fv[6]) - r, xmax = fmaxf(fmaxf(fv[0], fv[3]), fv[6]) + r;
                const float ymin = fminf(fminf(fv[1], fv[4]), fv[7]) - r, ymax = fmaxf(fmaxf(fv[1], fv[4]), fv[7]) + r;
                if (p.x > xmax || p.x < xmin || p.y > ymax || p.y < ymin) continue;
                const FaceEval e = eval_face(p, fv);
                if (e.pz < 0.0f) continue;                      // behind the image plane
                if (!e.inside && e.dist >= blur) continue;      // outside the blur band
                if (cnt == K && !(e.pz < zbuf[row + K - 1])) continue;  // farther than everything kept
                // stable sorted insertion: after every kept entry with depth <= pz
                int j = cnt < K ? cnt : K - 1;
                while (j > 0 && zbuf[row + j - 1] > e.pz) {
                    zbuf[row + j] = zbuf[row + j - 1];
                    pix_to_face[row + j] = pix_to_face[row + j - 1];
                    --j;
                }
                zbuf[row + j] = e.pz;
                pix_to_face[row + j] = f_begin + s_face[i];
                if (cnt < K) ++cnt;
            }
        }
    }
    // ---- bary / dists of the kept faces, then the padding of the warp's 32 rows as coalesced stores ----------
    if (in_image) {
#pragma unroll 1
        for (int k = 0; k < cnt; ++k) {
            const int64_t f = pix_to_face[row + k];
            float v[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) v[i] = __ldg(rs.face_verts + f * 9 + i);
            const FaceEval e = eval_face(p, v);
            bary[(row + k) * 3] = e.w0;
            bary[(row + k) * 3 + 1] = e.w1;
            bary[(row + k) * 3 + 2] = e.w2;
            dists[row + k] = e.inside ? -e.dist : e.dist;
        }
    }
    __syncthreads();
    s_face[threadIdx.x] = in_image ? cnt : K;  // kept count of every pixel of the tile (the face list is done with)
    __syncwarp();
    const int* const cnt_w = s_face + warp * 32;
    const int64_t wrow = (((int64_t)n * H + py) * W + blockIdx.x * TW) * K;  // first entry of the warp's rows
    if (py < H) {
        const int npix = min(TW, W - blockIdx.x * TW);
#pragma unroll 1
        for (int q = 0; q < npix; ++q) {
            const int c = cnt_w[q];
            const int64_t r0 = wrow + (int64_t)q * K;
#pragma unroll 1
            for (int k = c + lane; k < K; k += 32) {
                pix_to_face[r0 + k] = -1;
                zbuf[r0 + k] = -1.0f;
                dists[r0 + k] = -1.0f;
            }
#pragma unroll 1
            for (int j = 3 * c + lane; j < 3 * K; j += 32) bary[r0 * 3 + j] = -1.0f;
        }
    }
}


// Fast path for K <= KMAX: the K-buffer of a pixel is an array of packed 64-bit keys (depth bits << 32 | face)
// in SHARED memory, unsorted while the faces are walked and ranked at the end.  Depths are >= 0, so the integer order of
// the keys is the depth order with ties in face order; local memory is interleaved per thread, so the accesses of a warp
// are coalesced (the per-pixel output rows of the generic kernel are K*4 bytes apart: every shift of its sorted
// insertion was its own sector, 2.2 ms at config 2).
//
// WIDE: the bins are the bounded layout of pert_rasterize_bin_bounded: the tile walks its own list, then its image's wide
// list (bin num_bins + n), as one run of positions [f_lo, f_hi) whose tail is remapped into the wide list.
template <int KMAX, bool WIDE>
__global__ void __launch_bounds__(RT) rasterize_fwd_keys_kernel(const pert_raster rs, int64_t* __restrict__ pix_to_face,
                                                                float* __restrict__ zbuf, float* __restrict__ bary,
                                                                float* __restrict__ dists) {
    __shared__ float s_v[RT][9];
    __shared__ float4 s_bb[RT];  // bounding box grown by sqrt(blur_radius): xmin, xmax, ymin, ymax
    __shared__ int s_face[RT];
    __shared__ int s_wcount[RT / 32];
    const int H = rs.H, W = rs.W, K = rs.K;
    const int n = blockIdx.z, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int px = blockIdx.x * TW + lane, py = blockIdx.y * TH + warp;
    const bool in_image = px < W && py < H;
    const P2 p{pix_to_ndc(W - 1 - px, W, H), pix_to_ndc(H - 1 - py, H, W)};
    const int px0 = blockIdx.x * TW, px1 = min(px0 + TW, W) - 1, py0 = blockIdx.y * TH, py1 = min(py0 + TH, H) - 1;
    const float tx_hi = pix_to_ndc(W - 1 - px0, W, H), tx_lo = pix_to_ndc(W - 1 - px1, W, H);
    const float ty_hi = pix_to_ndc(H - 1 - py0, H, W), ty_lo = pix_to_ndc(H - 1 - py1, H, W);
    const float blur = rs.blur_radius, r = sqrtf(blur);
    const int64_t f_begin = __ldg(rs.face_start + n), f_end = __ldg(rs.face_start + n + 1);
    // the K-buffers of the tile's pixels live in SHARED memory, key j of thread t at [j * RT + t] (conflict-free).
    // As per-thread local arrays (512 B x 1024 resident threads per SM) they did not fit the L1 and thrashed to DRAM:
    // 2.6 GB of traffic for 0.73 GB of output, the rank loop at 46 % of the stall samples.
    extern __shared__ __align__(16) unsigned long long s_keys[];
    unsigned long long* const keys = s_keys + threadIdx.x;
    unsigned long long max_key = 0ull;
    int cnt = 0, max_idx = 0;
    // the faces this tile walks: its own bin (pert_rasterize_bin), or all faces of the mesh, in the caller's order
    // (nearest first when face_order is given: the sorted insertion below then appends almost always).  The result
    // does not depend on the order: keys are unique.
    const int64_t* const fmap = rs.bin_faces ? rs.bin_faces : rs.face_order;
    int64_t f_lo = f_begin, f_hi = f_end;
    int64_t f_split = 0, f_jump = 0;  // WIDE: positions >= f_split read bin_faces[position + f_jump]
    if (rs.bin_faces) {
        const int64_t bin = ((int64_t)n * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
        f_lo = __ldg(rs.bin_offset + bin);
        f_hi = f_lo + __ldg(rs.bin_count + bin);
        if (WIDE) {
            const int64_t wide = (int64_t)gridDim.z * gridDim.y * gridDim.x + n;
            f_split = f_hi;
            f_jump = __ldg(rs.bin_offset + wide) - f_split;
            f_hi += __ldg(rs.bin_count + wide);
        }
    }

#pragma unroll 1
    for (int64_t fc = f_lo; fc < f_hi; fc += RT) {
        const int64_t fpos = fc + threadIdx.x;
        int64_t f = fpos;
        bool keep = false;
        float v[9];
        float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
        if (fpos < f_hi) {
            if (fmap) f = __ldg(fmap + (WIDE && fpos >= f_split ? fpos + f_jump : fpos));
#pragma unroll
            for (int i = 0; i < 9; ++i) v[i] = __ldg(rs.face_verts + f * 9 + i);
            bb = make_float4(fminf(fminf(v[0], v[3]), v[6]) - r, fmaxf(fmaxf(v[0], v[3]), v[6]) + r,
                             fminf(fminf(v[1], v[4]), v[7]) - r, fmaxf(fmaxf(v[1], v[4]), v[7]) + r);
            const float zmax = fmaxf(fmaxf(v[2], v[5]), v[8]);
            const float area = edge(P2{v[0], v[1]}, P2{v[3], v[4]}, P2{v[6], v[7]});
            const bool zero_area = area <= kEps && area >= -kEps;
            const bool back = (rs.flags & PERT_RAST_CULL_BACKFACES) && area < 0.0f;
            keep = !(zmax < 0.0f) && !zero_area && !back && !(tx_lo > bb.y || tx_hi < bb.x || ty_lo > bb.w || ty_hi < bb.z);
        }
        const unsigned b = __ballot_sync(FULL, keep);
        if (lane == 0) s_wcount[warp] = __popc(b);
        __syncthreads();
        int base = 0, total = 0;
#pragma unroll
        for (int w = 0; w < RT / 32; ++w) {
            const int c = s_wcount[w];
            base += w < warp ? c : 0;
            total += c;
        }
        if (keep) {
            const int pos = base + __popc(b & ((1u << lane) - 1u));
            s_face[pos] = (int)(f - f_begin);
            s_bb[pos] = bb;
#pragma unroll
            for (int i = 0; i < 9; ++i) s_v[pos][i] = v[i];
        }
        __syncthreads();
        if (in_image) {
#pragma unroll 1
            for (int i = 0; i < total; ++i) {
                const float4 q = s_bb[i];
                if (p.x > q.y || p.x < q.x || p.y > q.w || p.y < q.z) continue;
                const float* fv = s_v[i];
                const P2 v0{fv[0], fv[1]}, v1{fv[3], fv[4]}, v2{fv[6], fv[7]};
                // the same arithmetic as eval_face, so the values recomputed for the kept faces are these
                const float area = edge(v2, v0, v1) + kEps;
                const float w0 = edge(p, v1, v2) / area, w1 = edge(p, v2, v0) / area, w2 = edge(p, v0, v1) / area;
                float pz = w0 * fv[2] + w1 * fv[5] + w2 * fv[8];
                if (pz < 0.0f) continue;
                if (!(w0 > 0.0f && w1 > 0.0f && w2 > 0.0f)) {  // outside the face: inside the blur band?
                    float tt;
                    bool dg;
                    const float d = fminf(fminf(point_line(p, v0, v1, tt, dg), point_line(p, v0, v2, tt, dg)),
                                          point_line(p, v1, v2, tt, dg));
                    if (d >= blur) continue;
                }
                if (pz == 0.0f) pz = 0.0f;  // -0 would sort last
                const unsigned long long key = ((unsigned long long)__float_as_uint(pz) << 32) | (unsigned)s_face[i];
                // UNSORTED buffer: appending is one store.  (A sorted insertion is a chain of dependent local-memory
                // loads, ~17 per candidate at 35 candidates: 43 % of the kernel's stall samples.)  Once the buffer is
                // full the farthest kept key is tracked and replaced; the order is established at the end by ranks.
                if (cnt < K) {
                    keys[(cnt++) * RT] = key;
                    if (cnt == K) {  // buffer just filled: find the farthest key (independent loads)
                        max_key = 0ull;
                        for (int j = 0; j < K; ++j)
                            if (keys[(j) * RT] > max_key) {
                                max_key = keys[(j) * RT];
                                max_idx = j;
                            }
                    }
                } else if (key < max_key) {
                    keys[(max_idx) * RT] = key;
                    max_key = 0ull;
                    for (int j = 0; j < K; ++j)
                        if (keys[(j) * RT] > max_key) {
                            max_key = keys[(j) * RT];
                            max_idx = j;
                        }
                }
            }
        }
    }
    const int64_t row = (((int64_t)n * H + py) * W + px) * K;
    if (in_image) {
#pragma unroll 1
        for (int k = 0; k < cnt; ++k) {
            // output slot = rank of the key (keys are unique: depth bits, then face index): cnt independent loads
            const unsigned long long key = keys[(k) * RT];
            int rank = 0;
            for (int j = 0; j < cnt; ++j) rank += keys[(j) * RT] < key ? 1 : 0;
            const int64_t f = f_begin + (int64_t)(unsigned)(key & 0xffffffffull);
            float v[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) v[i] = __ldg(rs.face_verts + f * 9 + i);
            const FaceEval e = eval_face(p, v);
            pix_to_face[row + rank] = f;
            zbuf[row + rank] = e.pz;
            bary[(row + rank) * 3] = e.w0;
            bary[(row + rank) * 3 + 1] = e.w1;
            bary[(row + rank) * 3 + 2] = e.w2;
            dists[row + rank] = e.inside ? -e.dist : e.dist;
        }
    }
    __syncthreads();
    s_face[threadIdx.x] = in_image ? cnt : K;
    __syncwarp();
    const int* const cnt_w = s_face + warp * 32;
    const int64_t wrow = (((int64_t)n * H + py) * W + blockIdx.x * TW) * K;
    if (py < H) {
        const int npix = min(TW, W - blockIdx.x * TW);
#pragma unroll 1
        for (int q = 0; q < npix; ++q) {
            const int c = cnt_w[q];
            const int64_t r0 = wrow + (int64_t)q * K;
#pragma unroll 1
            for (int k = c + lane; k < K; k += 32) {
                pix_to_face[r0 + k] = -1;
                zbuf[r0 + k] = -1.0f;
                dists[r0 + k] = -1.0f;
            }
#pragma unroll 1
            for (int j = 3 * c + lane; j < 3 * K; j += 32) bary[r0 * 3 + j] = -1.0f;
        }
    }
}


// ---------------------------------------------------------------------------------------------------------
// coarse binning for large meshes: which faces can touch which 32x4 pixel tile
// ---------------------------------------------------------------------------------------------------------
// The tiles of face f (one thread per face): its image n and the tile rectangle [tx0, tx1] x [ty0, ty1] overlapped by
// its bounding box grown by sqrt(blur_radius) (conservative by a pixel).  False for a face outside the ranges of
// face_start, culled (behind the camera, zero area, back face when culling) or whose box misses the image.
__device__ __forceinline__ bool face_tiles(const pert_raster& rs, int64_t f, int& n, int& tx0, int& tx1, int& ty0, int& ty1) {
    // image of this face: last n with face_start[n] <= f
    int lo = 0, hi = (int)rs.N;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(rs.face_start + mid) <= f) lo = mid; else hi = mid;
    }
    n = lo;
    if (f < __ldg(rs.face_start + n) || f >= __ldg(rs.face_start + n + 1)) return false;
    float v[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) v[i] = __ldg(rs.face_verts + f * 9 + i);
    const float r = sqrtf(rs.blur_radius);
    const float xmin = fminf(fminf(v[0], v[3]), v[6]) - r, xmax = fmaxf(fmaxf(v[0], v[3]), v[6]) + r;
    const float ymin = fminf(fminf(v[1], v[4]), v[7]) - r, ymax = fmaxf(fmaxf(v[1], v[4]), v[7]) + r;
    const float zmax = fmaxf(fmaxf(v[2], v[5]), v[8]);
    const float area = edge(P2{v[0], v[1]}, P2{v[3], v[4]}, P2{v[6], v[7]});
    if (zmax < 0.0f || (area <= kEps && area >= -kEps) || ((rs.flags & PERT_RAST_CULL_BACKFACES) && area < 0.0f)) return false;
    const int H = rs.H, W = rs.W;
    // pixel index i (from the -X / -Y side) whose centre is x: x = -range + (2 i + 1) range / S.  The float indices
    // are clamped to [-2, S+1] before the conversion: a box reaching |x| ~ 2^32 / S or inf would otherwise saturate
    // the conversion at INT_MAX and overflow the +-1 below.  Every test that follows gives the same answer on the
    // clamped index.  A NaN bound clamps to the far end (fmaxf / fminf return the other operand), so it covers the
    // whole axis, as in the unbinned kernels, whose tile test never culls on a NaN.
    const float rx = W > H ? (float)W / (float)H : 1.0f, ry = H > W ? (float)H / (float)W : 1.0f;
    const float fx0 = floorf(((xmin + rx) * (float)W / rx - 1.0f) * 0.5f), fx1 = ceilf(((xmax + rx) * (float)W / rx - 1.0f) * 0.5f);
    const float fy0 = floorf(((ymin + ry) * (float)H / ry - 1.0f) * 0.5f), fy1 = ceilf(((ymax + ry) * (float)H / ry - 1.0f) * 0.5f);
    const int ix0 = (int)fminf(fmaxf(fx0, -2.0f), (float)(W + 1)) - 1, ix1 = (int)fmaxf(fminf(fx1, (float)(W + 1)), -2.0f) + 1;
    const int iy0 = (int)fminf(fmaxf(fy0, -2.0f), (float)(H + 1)) - 1, iy1 = (int)fmaxf(fminf(fy1, (float)(H + 1)), -2.0f) + 1;
    if (ix1 < 0 || iy1 < 0 || ix0 > W - 1 || iy0 > H - 1) return false;
    // image column = W-1-i, row = H-1-i
    const int cx0 = W - 1 - min(ix1, W - 1), cx1 = W - 1 - max(ix0, 0), cy0 = H - 1 - min(iy1, H - 1), cy1 = H - 1 - max(iy0, 0);
    tx0 = cx0 / TW, tx1 = cx1 / TW, ty0 = cy0 / TH, ty1 = cy1 / TH;
    return true;
}

// Every tile of face_tiles gets the face.  FILL = false counts (atomics into bin_count, zeroed by the caller);
// FILL = true appends the face to every such tile's list at bin_offset[bin] + cursor++ (bin_cursor zeroed by the
// caller).  The order inside a list is arbitrary; the packed-key K-buffer makes the fragments independent of it.
template <bool FILL>
__global__ void __launch_bounds__(256) rasterize_bin_kernel(const pert_raster rs, int32_t* __restrict__ bin_count,
                                                            const int64_t* __restrict__ bin_offset, int32_t* __restrict__ bin_cursor,
                                                            int64_t* __restrict__ bin_faces) {
    const int64_t f = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (f >= rs.num_faces) return;
    int n, tx0, tx1, ty0, ty1;
    if (!face_tiles(rs, f, n, tx0, tx1, ty0, ty1)) return;
    const int tiles_x = (rs.W + TW - 1) / TW, tiles_y = (rs.H + TH - 1) / TH;
    for (int ty = ty0; ty <= ty1; ++ty)
        for (int tx = tx0; tx <= tx1; ++tx) {
            const int64_t bin = ((int64_t)n * tiles_y + ty) * tiles_x + tx;
            if (FILL)
                bin_faces[__ldg(bin_offset + bin) + atomicAdd(bin_cursor + bin, 1)] = f;
            else
                atomicAdd(bin_count + bin, 1);
        }
}

// Bounded layout (pert_rasterize_bin_bounded): a face with at most RASTER_BIN_CAP tiles goes into those tiles' lists
// (bins [0, num_bins)), as above; a face with more goes once into its image's wide list, bin num_bins + n, which every
// tile of the image walks after its own.  So no face has more than RASTER_BIN_CAP entries, and the caller sizes
// bin_faces as RASTER_BIN_CAP * num_faces without reading the counts back.  A face whose box reaches +-inf or NaN
// covers a whole axis, so it is wide unless the image has at most RASTER_BIN_CAP tiles along that axis.
template <bool FILL>
__global__ void __launch_bounds__(256) rasterize_bin_bounded_kernel(const pert_raster rs, int32_t* __restrict__ bin_count,
                                                                    const int64_t* __restrict__ bin_offset,
                                                                    int32_t* __restrict__ bin_cursor, int64_t* __restrict__ bin_faces) {
    const int64_t f = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (f >= rs.num_faces) return;
    int n, tx0, tx1, ty0, ty1;
    if (!face_tiles(rs, f, n, tx0, tx1, ty0, ty1)) return;
    const int tiles_x = (rs.W + TW - 1) / TW, tiles_y = (rs.H + TH - 1) / TH;
    const auto put = [&](int64_t bin) {
        if (FILL)
            bin_faces[__ldg(bin_offset + bin) + atomicAdd(bin_cursor + bin, 1)] = f;
        else
            atomicAdd(bin_count + bin, 1);
    };
    if ((tx1 - tx0 + 1) * (ty1 - ty0 + 1) > RASTER_BIN_CAP) {
        put(rs.N * tiles_y * tiles_x + n);
        return;
    }
    for (int ty = ty0; ty <= ty1; ++ty)
        for (int tx = tx0; tx <= tx1; ++tx) put(((int64_t)n * tiles_y + ty) * tiles_x + tx);
}

// ---------------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------------
constexpr int BT = 128, BW = BT / 32, BCHUNK = 1024;

// d E(p; a, b) / d(a, b) times g, accumulated (p fixed)
__device__ __forceinline__ void edge_bwd(P2 p, P2 a, P2 b, float g, P2& ga, P2& gb) {
    ga.x += g * (p.y - b.y);
    ga.y += g * (b.x - p.x);
    gb.x += -g * (p.y - a.y);
    gb.y += g * (p.x - a.x);
}

// TABLE: one grid row of CTAs per image; the gradients of that image's faces are accumulated in a shared-memory table
// (tcap faces; faces beyond it fall back to global atomics) and flushed once per CTA.  Every valid entry adds nine
// floats to its face: on a 1280-face mesh that is 79 M atomics on 11 k addresses per 8-view batch, which bound the
// global-atomics version (0.8 ms at config 2).
template <bool TABLE, int NT>
__global__ void __launch_bounds__(NT, NT == 512 ? 2 : 1) rasterize_bwd_kernel(const pert_raster rs, const int64_t* __restrict__ pix_to_face,
                                                           const float* __restrict__ grad_zbuf,
                                                           const float* __restrict__ grad_bary,
                                                           const float* __restrict__ grad_dists,
                                                           float* __restrict__ grad_face_verts, int64_t E, int64_t nchunks,
                                                           int tcap) {
    extern __shared__ __align__(16) float s_table[];  // TABLE: tcap * 9 floats, then the warps' valid lists
    constexpr int NWARP = NT / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t* const vlist = reinterpret_cast<uint16_t*>(s_table + (TABLE ? (size_t)tcap * 9 : 0)) + (size_t)warp * BCHUNK;
    const int H = rs.H, W = rs.W, K = rs.K;
    // TABLE: the chunks of image blockIdx.y, shared by the gridDim.x CTAs of that image; else all chunks, all CTAs
    const int64_t img_E = (int64_t)H * W * K;
    const int64_t e_first = TABLE ? (int64_t)blockIdx.y * img_E : 0, e_last = TABLE ? e_first + img_E : E;
    const int64_t my_chunks = TABLE ? (img_E + BCHUNK - 1) / BCHUNK : nchunks;
    int64_t f_begin = 0;
    if (TABLE) {
        f_begin = __ldg(rs.face_start + blockIdx.y);
        for (int i = threadIdx.x; i < tcap * 9; i += NT) s_table[i] = 0.0f;
        __syncthreads();
    }
    const int64_t w0 = (int64_t)blockIdx.x * NWARP + warp, wstride = (int64_t)gridDim.x * NWARP;
#pragma unroll 1
    for (int64_t c = w0; c < my_chunks; c += wstride) {
        const int64_t e_base = e_first + c * BCHUNK;
        const int Ec = (int)min((int64_t)BCHUNK, e_last - e_base);
        const int vec_ok = ((uintptr_t)(pix_to_face + e_base) & 15) == 0;
        const int nv = scan_valid(pix_to_face + e_base, Ec, vec_ok, vlist, BCHUNK);
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < nv; i += 32) {
            const int64_t e = e_base + vlist[i];
            const float gz = grad_zbuf ? __ldg(grad_zbuf + e) : 0.0f;
            const float gd_signed = grad_dists ? __ldg(grad_dists + e) : 0.0f;
            float gb0 = 0.f, gb1 = 0.f, gb2 = 0.f;
            if (grad_bary) {
                gb0 = __ldg(grad_bary + e * 3);
                gb1 = __ldg(grad_bary + e * 3 + 1);
                gb2 = __ldg(grad_bary + e * 3 + 2);
            }
            if (gz == 0.0f && gd_signed == 0.0f && gb0 == 0.0f && gb1 == 0.0f && gb2 == 0.0f) continue;
            const int64_t f = __ldg(pix_to_face + e);
            float v[9];
#pragma unroll
            for (int j = 0; j < 9; ++j) v[j] = __ldg(rs.face_verts + f * 9 + j);
            const int64_t pix = e / K;
            const int x = (int)(pix % W), y = (int)((pix / W) % H);
            const P2 p{pix_to_ndc(W - 1 - x, W, H), pix_to_ndc(H - 1 - y, H, W)};
            const P2 v0{v[0], v[1]}, v1{v[3], v[4]}, v2{v[6], v[7]};
            const FaceEval o = eval_face(p, v);
            P2 g0{0.f, 0.f}, g1{0.f, 0.f}, g2{0.f, 0.f};
            // pz = sum w_i z_i; w_i = e_i / area
            const float gw0 = gb0 + gz * v[2], gw1 = gb1 + gz * v[5], gw2 = gb2 + gz * v[8];
            const float inv_area = 1.0f / o.area;
            edge_bwd(p, v1, v2, gw0 * inv_area, g1, g2);  // e0 = E(p; v1, v2)
            edge_bwd(p, v2, v0, gw1 * inv_area, g2, g0);  // e1 = E(p; v2, v0)
            edge_bwd(p, v0, v1, gw2 * inv_area, g0, g1);  // e2 = E(p; v0, v1)
            // area = E(v2; v0, v1) + eps
            const float g_area = -(gw0 * o.w0 + gw1 * o.w1 + gw2 * o.w2) * inv_area;
            edge_bwd(v2, v0, v1, g_area, g0, g1);
            g2.x += g_area * (v1.y - v0.y);
            g2.y += -g_area * (v1.x - v0.x);
            // dists = +-|p - proj|^2 on the closest edge; the parameter's own derivative drops out (p - proj is
            // orthogonal to the edge where the clamp is inactive)
            if (gd_signed != 0.0f) {
                const float gd = o.inside ? -gd_signed : gd_signed;
                const P2 a = o.min_edge == 2 ? v1 : v0, b = o.min_edge == 0 ? v1 : v2;
                float tt;
                bool dg;
                point_line(p, a, b, tt, dg);
                const P2 proj{a.x + tt * (b.x - a.x), a.y + tt * (b.y - a.y)};
                const P2 rr = dg ? p - b : p - proj;
                const float ca = dg ? 0.0f : -2.0f * (1.0f - tt) * gd, cb = dg ? -2.0f * gd : -2.0f * tt * gd;
                P2& ga = o.min_edge == 2 ? g1 : g0;
                P2& gbb = o.min_edge == 0 ? g1 : g2;
                ga.x += ca * rr.x;
                ga.y += ca * rr.y;
                gbb.x += cb * rr.x;
                gbb.y += cb * rr.y;
            }
            const int64_t fl = f - f_begin;
            const float gv[9] = {g0.x, g0.y, gz * o.w0, g1.x, g1.y, gz * o.w1, g2.x, g2.y, gz * o.w2};
            // two code paths: a shared-memory atomic and a global one (a pointer selected at run time would make
            // every add a generic-address atomic)
            if (TABLE && fl >= 0 && fl < tcap) {
#pragma unroll
                for (int j = 0; j < 9; ++j) atomicAdd(s_table + fl * 9 + j, gv[j]);
            } else {
#pragma unroll
                for (int j = 0; j < 9; ++j) atomicAdd(grad_face_verts + f * 9 + j, gv[j]);
            }
        }
        __syncwarp();
    }
    if (TABLE) {
        __syncthreads();
        const int64_t nf = min((int64_t)tcap, __ldg(rs.face_start + blockIdx.y + 1) - f_begin);
        for (int i = threadIdx.x; i < nf * 9; i += NT)
            if (s_table[i] != 0.0f) atomicAdd(grad_face_verts + f_begin * 9 + i, s_table[i]);
    }
}

}  // namespace

int launch_rasterize_bin(const pert_raster& rs, int32_t* bin_count, const int64_t* bin_offset, int32_t* bin_cursor,
                         int64_t* bin_faces, cudaStream_t st) {
    const unsigned grid = (unsigned)((rs.num_faces + 255) / 256);
    if (bin_faces)
        rasterize_bin_kernel<true><<<grid, 256, 0, st>>>(rs, bin_count, bin_offset, bin_cursor, bin_faces);
    else
        rasterize_bin_kernel<false><<<grid, 256, 0, st>>>(rs, bin_count, bin_offset, bin_cursor, bin_faces);
    return (int)cudaGetLastError();
}

int launch_rasterize_bin_bounded(const pert_raster& rs, int32_t* bin_count, const int64_t* bin_offset, int32_t* bin_cursor,
                                 int64_t* bin_faces, cudaStream_t st) {
    const unsigned grid = (unsigned)((rs.num_faces + 255) / 256);
    if (bin_faces)
        rasterize_bin_bounded_kernel<true><<<grid, 256, 0, st>>>(rs, bin_count, bin_offset, bin_cursor, bin_faces);
    else
        rasterize_bin_bounded_kernel<false><<<grid, 256, 0, st>>>(rs, bin_count, bin_offset, bin_cursor, bin_faces);
    return (int)cudaGetLastError();
}

template <bool WIDE>
static cudaError_t launch_keys(const pert_raster& rs, dim3 grid, int64_t* pix_to_face, float* zbuf, float* bary, float* dists,
                               cudaStream_t st) {
    const size_t smem = (size_t)rs.K * RT * sizeof(unsigned long long);  // K = 50: 50 KB
    cudaError_t e = cudaFuncSetAttribute(rasterize_fwd_keys_kernel<64, WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    rasterize_fwd_keys_kernel<64, WIDE><<<grid, RT, smem, st>>>(rs, pix_to_face, zbuf, bary, dists);
    return cudaSuccess;
}

int launch_rasterize_fwd(const pert_raster& rs, int64_t* pix_to_face, float* zbuf, float* bary, float* dists, cudaStream_t st) {
    const dim3 grid((unsigned)((rs.W + TW - 1) / TW), (unsigned)((rs.H + TH - 1) / TH), (unsigned)rs.N);
    if (rs.K <= 64) {
        const cudaError_t e = rs.bin_faces && (rs.flags & PERT_RAST_BIN_WIDE)
                                  ? launch_keys<true>(rs, grid, pix_to_face, zbuf, bary, dists, st)
                                  : launch_keys<false>(rs, grid, pix_to_face, zbuf, bary, dists, st);
        if (e != cudaSuccess) return (int)e;
    } else  // K-buffer in the pixel's own output rows
        rasterize_fwd_rows_kernel<<<grid, RT, 0, st>>>(rs, pix_to_face, zbuf, bary, dists);
    return (int)cudaGetLastError();
}

int launch_rasterize_bwd(const pert_raster& rs, const int64_t* pix_to_face, const float* grad_zbuf, const float* grad_bary,
                         const float* grad_dists, float* grad_face_verts, cudaStream_t st) {
    const int64_t E = (int64_t)rs.N * rs.H * rs.W * rs.K, nchunks = (E + BCHUNK - 1) / BCHUNK;
    constexpr int NT = 512;
    const int64_t per_mesh = (rs.num_faces + rs.N - 1) / rs.N;  // exact for a batch of poses of one topology
    const int tcap = (int)(per_mesh < 4096 ? per_mesh : 4096);
    const size_t smem = (size_t)tcap * 9 * sizeof(float) + (size_t)(NT / 32) * BCHUNK * sizeof(uint16_t);
    const int64_t img_chunks = ((int64_t)rs.H * rs.W * rs.K + BCHUNK - 1) / BCHUNK;
    if (img_chunks >= 4 * (NT / 32)) {  // enough entries per image for a table to pay
        cudaError_t e = cudaFuncSetAttribute(rasterize_bwd_kernel<true, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        int per_sm = (int)((200 * 1024) / smem);
        per_sm = per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm);
        int64_t ctas = (sm_count() * (int64_t)per_sm + rs.N - 1) / rs.N;
        const int64_t most = (img_chunks + NT / 32 - 1) / (NT / 32);
        if (ctas > most) ctas = most;
        rasterize_bwd_kernel<true, NT><<<dim3((unsigned)ctas, (unsigned)rs.N), NT, smem, st>>>(
            rs, pix_to_face, grad_zbuf, grad_bary, grad_dists, grad_face_verts, E, nchunks, tcap);
    } else {
        const int64_t cap = sm_count() * 8, need = (nchunks + BW - 1) / BW;
        rasterize_bwd_kernel<false, BT><<<(unsigned)(need < cap ? need : cap), BT, (size_t)BW * BCHUNK * sizeof(uint16_t), st>>>(
            rs, pix_to_face, grad_zbuf, grad_bary, grad_dists, grad_face_verts, E, nchunks, 0);
    }
    return (int)cudaGetLastError();
}

}  // namespace pert
