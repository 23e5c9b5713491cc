// Host-side launch interface between the C ABI (cabi.cu) and the kernel translation units.
#pragma once
#include "common.cuh"

namespace pert {

struct FwdArgs {
    pert_problem pb;
    Launch L;
    float* image;
    uint16_t* counts;
    float* rsum;
    void* winners;
    uint16_t* pixstate;
    int32_t* hist;
    int32_t* worklist;  // [0] = number of tiles handed to the fallback pass, [4..] = their indices
    int32_t* blob;      // tile blobs written by the sparse-first main pass (see common.cuh), or NULL
};

struct BwdArgs {
    pert_problem pb;
    Launch L;
    const float* grad_image;
    const uint16_t* counts;
    const float* rsum;
    const void* winners;
    const uint16_t* pixstate;
    float* grad_dists;
    float* grad_zbuf;
    float* grad_colors;
    float* partials;
    float* acc;
    float* pixstat;
    const int32_t* hist;
    int32_t* worklist;
    const int32_t* blob;  // tile blobs of forward, or NULL: backward then rescans and recomputes
};

int fwd_smem_layout(int tp, int cap, SmemLayout& L);  // returns the bytes the coverage-sample phase needs
void bwd_smem_layout(int tp, int K, int cap, int sc, int nchunks, int win_bytes, bool compact, bool lean, SmemLayout& L);

// return a cudaError_t as int (0 = success)
// `fb` (optional): launch record of the fallback pass of the sparse-first mode (half-size tiles)
int launch_shade_fwd(const FwdArgs& a, const FwdArgs* fb, cudaStream_t st);
int launch_shade_bwd(const BwdArgs& a, const BwdArgs* fb, float* grad_scalars, cudaStream_t st);
// forward-only render: image only (a.counts = the fallback pass's workspace or NULL; no other saved state); with one phase
// bit (pert_shade_render_phase) a.counts / a.hist are that phase's inputs and outputs
int launch_shade_render(const FwdArgs& a, const FwdArgs* fb, cudaStream_t st);

void soft_smem_layout(int tp, int K, bool bwd, SmemLayout& L);
int launch_soft_fwd(const pert_problem& pb, const Launch& L, float* image, cudaStream_t st);
int launch_soft_bwd(const pert_problem& pb, const Launch& L, const float* grad_image, float* grad_dists, float* grad_zbuf,
                    float* grad_colors, float* partials, float* grad_scalars, cudaStream_t st);

int launch_rast_fwd(const float* x, int64_t P, int K, int S, int s_begin, int s_end, float sigma, uint64_t seed,
                    int64_t pixel_offset, const float* noise, uint32_t flags, float* prob, float* rsum, cudaStream_t st);
int launch_rast_bwd(const float* grad_l, const float* rsum, int64_t n, int S, float sigma, float* grad_x,
                    float* partials, float* grad_sigma, cudaStream_t st);
int launch_argmax_fwd(const float* z, int64_t P, int K1, int S, int s_begin, int s_end, float gamma, uint64_t seed,
                      int64_t pixel_offset, const float* noise, uint32_t flags, float* weights, void* winners,
                      cudaStream_t st);
int launch_argmax_bwd(const float* grad_l, const float* z, const void* winners, int64_t P, int K1, int S, int s_begin,
                      int s_end, float gamma, uint64_t seed, int64_t pixel_offset, const float* noise, uint32_t flags,
                      float* grad_z, float* partials, float* grad_gamma, cudaStream_t st);
// atlas != NULL: the texel source is the (num_faces, atlas_r, atlas_r, 3) atlas (pert_phong_atlas_fwd / _bwd), and
// grad_texels is its gradient
int launch_phong_fwd(const pert_phong& ph, float* colors, cudaStream_t st, const float* atlas = nullptr, int atlas_r = 0);
int launch_phong_bwd(const pert_phong& ph, const float* grad_colors, float* grad_texels, float* grad_bary, float* grad_fv,
                     float* grad_fn, cudaStream_t st, const float* atlas = nullptr, int atlas_r = 0);
int launch_phong_light_bwd(const pert_phong& ph, const float* grad_colors, float* grad_lighting, cudaStream_t st,
                           const float* atlas = nullptr, int atlas_r = 0);
// most tile entries of one face in the bounded bins of pert_rasterize_bin_bounded (csrc/raster.cu); chosen by
// measurement among 4, 8 and 16 (profiles/r10_raster_bins.txt; the others built with -DPERT_RASTER_BIN_CAP=C)
#ifndef PERT_RASTER_BIN_CAP
#define PERT_RASTER_BIN_CAP 8
#endif
constexpr int RASTER_BIN_CAP = PERT_RASTER_BIN_CAP;
int launch_rasterize_bin_bounded(const pert_raster& rs, int32_t* bin_count, const int64_t* bin_offset, int32_t* bin_cursor,
                                 int64_t* bin_faces, cudaStream_t st);
int launch_rasterize_bin(const pert_raster& rs, int32_t* bin_count, const int64_t* bin_offset, int32_t* bin_cursor,
                         int64_t* bin_faces, cudaStream_t st);
int launch_rasterize_fwd(const pert_raster& rs, int64_t* pix_to_face, float* zbuf, float* bary, float* dists, cudaStream_t st);
int launch_rasterize_bwd(const pert_raster& rs, const int64_t* pix_to_face, const float* grad_zbuf, const float* grad_bary,
                         const float* grad_dists, float* grad_face_verts, cudaStream_t st);
int launch_seed_advance(uint64_t* seed_device, cudaStream_t st);
int launch_noise_fill(uint64_t seed, int stage, int64_t P, int slots, int s_begin, int s_end, int64_t pixel_offset,
                      float* out, cudaStream_t st);

}  // namespace pert
