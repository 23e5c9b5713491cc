"""The chunked oracle of the whole-image checks (test_gpu_timed_instantiation.chunked_shade_fwd_bwd) equals one call of
O.shade_fwd_bwd on the whole problem: chunk offsets, noise slices, concatenation and the float64 scalar sums."""

import torch

from oracle import pert_oracle as O
from test_gpu_timed_instantiation import ALPHA, BG, EPS, GAMMA, SIGMA, chunked_shade_fwd_bwd


def test_chunked_oracle_equals_the_one_shot_oracle():
    import pertrenderer_b200 as pb
    N, HW, K, S = 2, 6, 5, 8
    P = N * HW * HW
    fr, col = pb.synthetic_fragments(N, HW, HW, K, kind="realistic", sigma=SIGMA, seed=3, device="cpu", coverage=0.8)
    gen = torch.Generator().manual_seed(4)
    U = torch.randn((S, N, HW, HW, K), generator=gen)
    V = torch.randn((S, N, HW, HW, K + 1), generator=gen)
    G = torch.randn((N, HW, HW, 4), generator=gen)
    st, gr = O.shade_fwd_bwd(fr.pix_to_face, fr.zbuf, fr.dists, col, BG, 1.0, 100.0, SIGMA, GAMMA, ALPHA, EPS, U, V, G)
    assert (st.counts > 0).any() and (st.a_s != st.a_0).any() and gr["dists"].abs().max() > 0  # not a vacuous case

    def noise(c0, n):  # the generator's tensors sliced the way noise_fill(..., pixel_offset=c0) slices the Philox stream
        return U.reshape(S, P, K)[:, c0:c0 + n].reshape(S, 1, 1, n, K), V.reshape(S, P, K + 1)[:, c0:c0 + n].reshape(S, 1, 1, n, K + 1)

    flat = lambda t, tail: t.reshape((P,) + tail)  # noqa: E731
    for chunk in (7, 32, P):  # uneven last chunk, several chunks, one
        out = chunked_shade_fwd_bwd(flat(fr.pix_to_face, (K,)), flat(fr.zbuf, (K,)), flat(fr.dists, (K,)), flat(col, (K, 3)),
                                    flat(G, (4,)), noise, chunk)
        assert torch.equal(out["counts"], flat(st.counts, (K,)))
        assert torch.equal(out["a_s"], st.a_s.reshape(S, P))
        assert torch.equal(out["image"], flat(st.image, (4,)))
        for k, tail in (("dists", (K,)), ("zbuf", (K,)), ("colors", (K, 3))):
            assert torch.allclose(out[k], flat(gr[k], tail), rtol=1e-6, atol=1e-6 * gr[k].abs().max().item()), (chunk, k)
        for k in ("sigma", "gamma", "alpha"):
            assert isinstance(out[k], float)
            assert abs(out[k] - gr[k].item()) <= 1e-5 * abs(gr[k].item()) + 1e-9, (chunk, k, out[k], gr[k].item())
