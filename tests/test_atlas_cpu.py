"""Texture atlases without a GPU: the atlas Phong entry points (pert_phong_atlas_fwd / _bwd) are exported and bound once,
every refusal of their argument validation comes before any device work, a library built before them is refused with a
request to rebuild, and AtlasTexels.materialize follows the cell rule of include/pertshade.h -- checked against a NumPy
restatement, and against pytorch3d's rule wherever that rule picks an in-range cell.  No call here launches a kernel:
the pointers are fake."""

import types

import numpy as np
import pytest
import torch

from pertrenderer_b200 import _cabi
from pertrenderer_b200.structures import AtlasTexels

FAKE = 1 << 20  # aligned, never dereferenced


def _phong(unlit=False, F=4):
    ph = _cabi.PertPhong()
    ph.P, ph.HW, ph.K, ph.num_faces, ph.light_rows = 8, 4, 2, F, 1
    ph.flags = _cabi.PHONG_UNLIT if unlit else 0
    ph.pix_to_face = ph.bary = FAKE
    if not unlit:
        ph.face_verts = ph.face_normals = ph.lighting = FAKE
    return ph


def test_atlas_symbols_are_exported_and_bound_once():
    lib = _cabi.load()
    for name in ("pert_phong_atlas_fwd", "pert_phong_atlas_bwd"):
        assert hasattr(lib, name) and name in _cabi.EXPORTS
    fwd, bwd = _cabi.phong_atlas_fns()
    assert _cabi.phong_atlas_fns() == (fwd, bwd)
    assert _cabi.phong_atlas_fns()[0] is fwd and _cabi.phong_atlas_fns()[1] is bwd
    assert lib.pert_version() == _cabi.ABI_VERSION == 15


def test_library_without_atlas_kernels_is_refused(monkeypatch):
    """A library built before the atlas entry points keeps serving every other call; the first atlas call asks for a
    rebuild."""
    monkeypatch.setattr(_cabi, "_lib", types.SimpleNamespace())
    monkeypatch.setattr(_cabi, "_phong_atlas", None)
    with pytest.raises(_cabi.PertLibraryError, match="rebuild"):
        _cabi.phong_atlas_fns()


@pytest.mark.parametrize("unlit", [False, True])
def test_atlas_refusals(unlit):
    fwd, bwd = _cabi.phong_atlas_fns()
    f = FAKE
    ph = _phong(unlit)
    # every output NULL and no lighting gradient: validation passes and nothing is launched
    assert bwd(ph, f, 4, f, None, None, None, None, None, None) == 0
    assert fwd(None, f, 4, f, None) == -1
    assert bwd(None, f, 4, f, None, None, None, None, None, None) == -1
    assert fwd(ph, None, 4, f, None) == -1  # no atlas
    assert bwd(ph, None, 4, f, f, None, None, None, None, None) == -1
    assert fwd(ph, f, 4, None, None) == -1  # no colors
    assert bwd(ph, f, 4, None, f, None, None, None, None, None) == -1  # no grad_colors
    for field in ("texels", "face_colors", "face_vert_colors", "uv_map"):  # a second texel source
        ph = _phong(unlit)
        setattr(ph, field, f)
        if field == "uv_map":
            ph.face_uvs, ph.map_h, ph.map_w, ph.map_count = f, 4, 4, 1
        assert fwd(ph, f, 4, f, None) == -3, field
        assert bwd(ph, f, 4, f, f, f, None, None, None, None) == -3, field
    ph = _phong(unlit)
    for size in (0, -1, -(1 << 31)):
        assert fwd(ph, f, size, f, None) == -2, size
        assert bwd(ph, f, size, f, f, None, None, None, None, None) == -2, size
    # 32-bit atlas offsets: num_faces R^2 3 <= 2^31 - 1 (26754^2 3 = 2147329548 fits, 26755^2 3 = 2147490075 does not)
    one = _phong(unlit, F=1)
    assert fwd(one, f, 26755, f, None) == -3
    assert fwd(one, f, (1 << 31) - 1, f, None) == -3
    assert fwd(_phong(unlit, F=1000), f, 847, f, None) == -3  # 1000 847^2 3 = 2152227000
    assert fwd(one, f, 26754, f + 2, None) == -4  # accepted size: the misaligned colors are what is refused
    assert bwd(one, f, 26754, f, None, None, None, None, None, None) == 0
    # alignment
    assert fwd(ph, f + 2, 4, f, None) == -4
    assert bwd(ph, f + 2, 4, f, None, None, None, None, None, None) == -4
    assert bwd(ph, f, 4, f, f + 2, None, None, None, None, None) == -4  # grad_atlas
    assert bwd(ph, f, 4, f + 1, f, None, None, None, None, None) == -4
    assert bwd(ph, f, 4, f, None, f + 2, None, None, None, None) == -4
    # the shared rules of pert_phong_fwd / _bwd
    bad = _phong(unlit)
    bad.P = 0
    assert fwd(bad, f, 4, f, None) == -2
    bad = _phong(unlit)
    bad.pix_to_face = None
    assert fwd(bad, f, 4, f, None) == -1
    bad = _phong(unlit)
    bad.bary = f + 2
    assert fwd(bad, f, 4, f, None) == -4
    if unlit:  # no lighting gradient without lighting
        assert bwd(ph, f, 4, f, None, None, None, None, f, None) == -3
    else:
        bad = _phong(unlit)
        bad.face_normals = None
        assert fwd(bad, f, 4, f, None) == -1
        bad = _phong(unlit)
        bad.light_rows = 3
        assert fwd(bad, f, 4, f, None) == -2


def test_phong_without_a_texel_source_is_still_refused():
    lib = _cabi.load()
    ph = _phong()
    assert lib.pert_phong_fwd(ph, FAKE, None) == -1
    assert lib.pert_phong_bwd(ph, FAKE, None, None, None, None, None, None) == -1


# ---- the cell rule ----------------------------------------------------------------------------------------------------

def _special_values(R):
    """Barycentric coordinates in range, negative down to -3, above 1, exactly k/R, NaN and +-inf."""
    k = [np.float32(i) / np.float32(R) for i in range(R + 1)]
    neg = [-3.0, -2.5, -1.0, -0.75, -0.5, -1.0 / R, -0.5 / R, -1e-7, -0.0]
    above = [1.0, 1.0 + 1e-7, 1.25, 1.5, 2.0, 3.0, 1e6]
    inr = [0.1, 0.25, 0.3, 0.49, 0.5, 0.6, 0.7, 0.999]
    odd = [np.nan, np.inf, -np.inf, 3.4e38, -3.4e38]
    return np.array(k + neg + above + inr + odd, dtype=np.float32)


def _pairs(R, seed=0):
    v = _special_values(R)
    w0, w1 = np.meshgrid(v, v, indexing="ij")
    w0, w1 = w0.ravel(), w1.ravel()
    # points on the diagonal w0 + w1 = 1 and just off it, and random points in and around the triangle
    rng = np.random.default_rng(seed)
    t = rng.random(256).astype(np.float32)
    diag0 = np.concatenate([t, np.array([i / R for i in range(R + 1)], dtype=np.float32)])
    diag1 = (np.float32(1.0) - diag0).astype(np.float32)
    r = rng.uniform(-0.5, 1.5, size=(2, 512)).astype(np.float32)
    w0 = np.concatenate([w0, diag0, diag0, r[0]])
    w1 = np.concatenate([w1, diag1, np.nextafter(diag1, np.float32(2)), r[1]])
    return w0.astype(np.float32), w1.astype(np.float32)


def _numpy_cells(w0, w1, R):
    """include/pertshade.h's rule, restated in NumPy float32."""
    with np.errstate(over="ignore", invalid="ignore"):
        w0 = np.nan_to_num(w0, nan=0.0)
        w1 = np.nan_to_num(w1, nan=0.0)
        Rf = np.float32(R)
        wx = np.minimum(np.trunc(np.clip(w0 * Rf, np.float32(-1), Rf)).astype(np.int64), R - 1)
        wy = np.minimum(np.trunc(np.clip(w1 * Rf, np.float32(-1), Rf)).astype(np.int64), R - 1)
        s = (w0 + w1).astype(np.float32) * Rf
        below = (s.astype(np.float32) - (wx + wy).astype(np.float32)) <= np.float32(1)
    wx = np.clip(np.where(below, wx, R - 1 - wx), 0, R - 1)
    wy = np.clip(np.where(below, wy, R - 1 - wy), 0, R - 1)
    return wx, wy


def _parent_cells(w0, w1, R):
    """The rule before the unclipped coordinates were handled (pytorch3d's, with the cell clamped to R - 1), up to the
    index: cells outside [0, R) are what it wrapped or overflowed."""
    w01 = torch.stack([w0, w1], -1)
    w_xy = (w01 * R).to(torch.int64).clamp(max=R - 1)
    below = (w01.sum(dim=-1) * R - w_xy.to(w01.dtype).sum(dim=-1)) <= 1.0
    w_x, w_y = w_xy.unbind(-1)
    return torch.where(below, w_x, R - 1 - w_x), torch.where(below, w_y, R - 1 - w_y)


def _cell_atlas(F, R):
    """An atlas whose texel says where it is: texel [f, y, x] = (((f R + y) R + x) 3 + c)."""
    return torch.arange(F * R * R * 3, dtype=torch.float32).reshape(F, R, R, 3)


def _materialized_cells(w0, w1, R, F=3):
    n = w0.shape[0]
    face = torch.arange(n, dtype=torch.int64) % F
    p2f = face.reshape(1, 1, n, 1)
    bary = torch.stack([torch.from_numpy(w0), torch.from_numpy(w1), torch.full((n,), 0.5)], -1).reshape(1, 1, n, 1, 3)
    tex = AtlasTexels(_cell_atlas(F, R)).materialize(p2f, bary).reshape(n, 3)
    off = tex[:, 0].to(torch.int64) // 3 - face * R * R
    return (off % R).numpy(), (off // R).numpy()


@pytest.mark.parametrize("R", [1, 2, 3, 4, 8])
def test_materialize_follows_the_cell_rule(R):
    w0, w1 = _pairs(R)
    wx, wy = _materialized_cells(w0, w1, R)
    ex, ey = _numpy_cells(w0, w1, R)
    bad = np.nonzero((wx != ex) | (wy != ey))[0]
    assert bad.size == 0, [(w0[i], w1[i], (wx[i], wy[i]), (ex[i], ey[i])) for i in bad[:5]]


@pytest.mark.parametrize("R", [1, 2, 3, 4, 8])
def test_materialize_keeps_every_in_range_cell_of_the_old_rule(R):
    """Wherever the old rule picked an in-range cell without wrapping, the cell is the same; in-range coordinates
    ([0, 1], sums above 1 included) never wrapped."""
    w0, w1 = _pairs(R)
    fin = np.isfinite(w0) & np.isfinite(w1) & (np.abs(w0) < 1e6) & (np.abs(w1) < 1e6)
    w0, w1 = w0[fin], w1[fin]
    px, py = _parent_cells(torch.from_numpy(w0), torch.from_numpy(w1), R)
    px, py = px.numpy(), py.numpy()
    ok = (px >= 0) & (px < R) & (py >= 0) & (py < R)
    in_range = (w0 >= 0) & (w0 <= 1) & (w1 >= 0) & (w1 <= 1)
    assert ok[in_range].all()
    wx, wy = _materialized_cells(w0, w1, R)
    assert np.array_equal(wx[ok], px[ok]) and np.array_equal(wy[ok], py[ok])
    assert (~ok).any()  # the set holds coordinates the old rule wrapped or overflowed on


def test_materialize_padding_and_gradient():
    """Padded entries read zero whatever their coordinates; the gradient of an out-of-range coordinate lands in a cell
    of the grid."""
    R, F = 4, 2
    atlas = torch.rand(F, R, R, 3).requires_grad_(True)
    p2f = torch.tensor([[[[0, 1, -1]]]])
    bary = torch.tensor([[[[[-3.0, 0.5, 3.5], [2.5, -1.5, 0.0], [float("nan"), float("inf"), 0.0]]]]])
    tex = AtlasTexels(atlas).materialize(p2f, bary)
    assert (tex[0, 0, 0, 2] == 0).all()
    tex.sum().backward()
    assert atlas.grad.sum().item() == 6.0 and (atlas.grad.sum(-1) > 0).sum().item() == 2
