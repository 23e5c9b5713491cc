"""CPU oracle of the shader without control variates (GaussianRast_wovr + GaussianAgg_wovr, randomras/smoothrast.py:61-108
and randomras/smoothagg.py:75-141, eval.py:152-154 "gaussian_wovr"), test infrastructure only.  Forward is the Gaussian
oracle's (oracle/pert_oracle.py): the estimators change backward only.  Coverage uses sum_s h_s U_s instead of
sum_s (h_s - h0) U_s, aggregation c_s = g[a_s] instead of g[a_s] - g[a_0]; so samples that picked a_0, and pixels
without any valid entry (the background wins every sample), contribute too.  Pinned against the unmodified reference's
own draws and gradients by tests/test_wovr_cpu.py (tests/golden/ops_wovr.npz)."""

import torch

from oracle import pert_oracle as O

F32 = torch.float32


def shade_fwd_bwd(pix_to_face, zbuf, dists, colors, background, znear, zfar, sigma, gamma, alpha, eps, U, V, grad_image):
    """smooth_rgb_blend with GaussianRast_wovr + GaussianAgg_wovr fed with explicit draws U, V: (ShadeState, gradients)."""
    st = O.shade_forward(pix_to_face, zbuf, dists, colors, background, znear, zfar, sigma, gamma, alpha, eps, U, V)
    grad_w = O._grad_weights(colors, grad_image, st.aux["bg"])
    grad_zeta, grad_gamma = O.random_argmax_bwd(grad_w, st.a_s, st.a_0, V, gamma, control_variate=False)
    # mean_s h U / sigma: the coverage estimator's gradient for an upstream gradient of one
    cov, _ = O.random_heaviside_bwd(torch.ones_like(dists), st.h, st.h0, U, sigma, control_variate=False)
    return st, O._finish_backward(st.prob, st.weights, st.aux, grad_image, zbuf, colors, gamma, alpha, eps, grad_zeta,
                                  grad_gamma, cov)


# noise-sample shards: the per-shard sums without control variates; the finish from reduced sums is
# O.shade_backward_from_sums
def rast_shard_sums(dists, U_shard, sigma):
    """(hit counts, sum_s h U), both (N,H,W,K) float."""
    _, h, _ = O.random_heaviside_fwd(-dists, U_shard, sigma)
    return h.sum(dim=0), (h * U_shard).sum(dim=0)


def argmax_score_sums(grad_w, a_s, V_shard):
    """Packed (N,H,W,K1+2) with c_s = g[a_s]: [..., :K1] = sum_s c_s V_sj, [..., K1] = sum_s c_s ||V_s||^2,
    [..., K1+1] = sum_s c_s."""
    S = V_shard.shape[0]
    gl_s = grad_w.unsqueeze(0).expand(S, *grad_w.shape)
    c = torch.gather(gl_s, -1, a_s.unsqueeze(-1)).squeeze(-1)
    acc = (c.unsqueeze(-1) * V_shard).sum(dim=0)
    t2 = (c * (V_shard * V_shard).sum(dim=-1)).sum(dim=0)
    return torch.cat((acc, t2[..., None], c.sum(dim=0)[..., None]), dim=-1)
