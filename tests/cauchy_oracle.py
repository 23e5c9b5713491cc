"""CPU oracle of the Cauchy-perturbed shader (ArctanRast + CauchyAgg, randomras/smoothrast.py:162-173 and
randomras/smoothagg.py:230-250), test infrastructure only.  Forward is the Gaussian oracle's (oracle/pert_oracle.py) fed
with Cauchy draws: only the noise law changes.  Backward differs by the score of the noise density: every estimator
multiplies the noise n by psi(n) = 2n / (1 + n^2) instead of n (smoothrast.py:49-50, smoothagg.py:57-63), and the
gamma term uses sum_j V_sj psi(V_sj) where the Gaussian branch has ||V_s||^2.  Pinned against the unmodified reference's
own Cauchy draws and gradients by tests/test_cauchy_cpu.py (tests/golden/ops_cauchy.npz)."""

import torch

from oracle import pert_oracle as O

F32 = torch.float32


def score(n):
    """psi(n) = -d/dn log p(n) of the standard Cauchy density."""
    return 2.0 * n / (1.0 + n * n)


def random_heaviside_bwd(grad_l, h, h0, U, sigma):
    """smoothrast.py:40-59, cauchy branch: the Gaussian estimator with U replaced by psi(U)."""
    return O.random_heaviside_bwd(grad_l, h, h0, score(U), sigma)


def random_argmax_bwd(grad_l, a_s, a_0, V, gamma):
    """smoothagg.py:45-73, cauchy branch: grad_zeta_j = mean_s c_s psi(V_sj) / gamma for all j,
    grad_gamma = mean_s sum_pixels c_s (sum_j V_sj psi(V_sj) - 1) / gamma."""
    g = torch.as_tensor(gamma, dtype=F32)
    S = V.shape[0]
    gl_s = grad_l.unsqueeze(0).expand(S, *grad_l.shape)
    g_sel = torch.gather(gl_s, -1, a_s.unsqueeze(-1)).squeeze(-1)
    g_ref = torch.gather(grad_l, -1, a_0.unsqueeze(-1)).squeeze(-1)
    c = g_sel - g_ref.unsqueeze(0)
    psi = score(V)
    grad_zeta = (c.unsqueeze(-1) * psi / g).sum(dim=0) / S
    vpsi = (V * psi).sum(dim=-1)
    grad_gamma = (c * (vpsi - 1.0) / g).sum(dim=(1, 2, 3)).sum() / S
    return grad_zeta, grad_gamma


def shade_fwd_bwd(pix_to_face, zbuf, dists, colors, background, znear, zfar, sigma, gamma, alpha, eps, U, V, grad_image):
    """smooth_rgb_blend with ArctanRast + CauchyAgg fed with explicit Cauchy draws U, V: (ShadeState, gradient dict)."""
    st = O.shade_forward(pix_to_face, zbuf, dists, colors, background, znear, zfar, sigma, gamma, alpha, eps, U, V)
    grad_w = O._grad_weights(colors, grad_image, st.aux["bg"])
    grad_zeta, grad_gamma = random_argmax_bwd(grad_w, st.a_s, st.a_0, V, gamma)
    sig = torch.as_tensor(sigma, dtype=F32)
    cov = ((st.h - st.h0.unsqueeze(0)) * score(U) / sig).sum(dim=0) / U.shape[0]
    return st, O._finish_backward(st.prob, st.weights, st.aux, grad_image, zbuf, colors, gamma, alpha, eps, grad_zeta,
                                  grad_gamma, cov)


# noise-sample shards: the per-shard sums carry psi; the finish from reduced sums is O.shade_backward_from_sums
def rast_shard_sums(dists, U_shard, sigma):
    """(hit counts, sum_s (h - h0) psi(U)), both (N,H,W,K) float."""
    _, h, h0 = O.random_heaviside_fwd(-dists, U_shard, sigma)
    return h.sum(dim=0), ((h - h0.unsqueeze(0)) * score(U_shard)).sum(dim=0)


def argmax_score_sums(grad_w, a_s, a_0, V_shard):
    """Packed (N,H,W,K1+2): [..., :K1] = sum_s c_s psi(V_sj), [..., K1] = sum_s c_s sum_j V_sj psi(V_sj),
    [..., K1+1] = sum_s c_s."""
    S = V_shard.shape[0]
    gl_s = grad_w.unsqueeze(0).expand(S, *grad_w.shape)
    c = torch.gather(gl_s, -1, a_s.unsqueeze(-1)).squeeze(-1) - torch.gather(grad_w, -1, a_0.unsqueeze(-1)).squeeze(-1)
    psi = score(V_shard)
    acc = (c.unsqueeze(-1) * psi).sum(dim=0)
    t2 = (c * (V_shard * psi).sum(dim=-1)).sum(dim=0)
    return torch.cat((acc, t2[..., None], c.sum(dim=0)[..., None]), dim=-1)
