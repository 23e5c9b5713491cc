"""pert_blob_bytes (no GPU): the tile_blob buffer holds one tile blob per tile of the sparse-first main pass and then one
fallback record per half-tile of every tile (csrc/common.cuh), the worst case of every tile going to the fallback pass."""

import pytest

from pertrenderer_b200 import _cabi

SMS = 148  # the tile geometry of small jobs follows the SM count: a B200's, and what the library assumes without a GPU


def _sparse_tp(K, P):
    base = 32 if K <= 16 else 16 if K <= 32 else 8 if K <= 64 else 4
    tp = min(2 * base, 32)
    if tp > base and (P + tp - 1) // tp < SMS * 24:
        tp = base
    while tp > 4 and (P + tp - 1) // tp < SMS * 16:
        tp >>= 1
    return tp


def _words(n):
    return (n + 3) & ~3


def _expected(N, H, W, K):
    P = N * H * W
    tp = _sparse_tp(K, P)
    cap = max(32, (tp * K // 5 + 7) & ~7)
    if cap > tp * K:
        cap = (tp * K + 1) & ~1
    tiles = (P + tp - 1) // tp
    blob = _words(2 + 7 * tp + 2 * cap)                  # nv, vstart, 6 per pixel, vlist + counts (u16), zeta
    h, hcap = tp // 2, tp // 2 * K
    record = _words(2 + 7 * h + hcap // 2 + hcap)        # nv, vstart, 6 per pixel, vlist (u16), zeta
    return tp, 4 * (tiles * blob + 2 * tiles * record)


@pytest.mark.parametrize("shape, tp", [
    ((8, 256, 256, 50), 16),   # BASELINE config 2
    ((2, 128, 128, 100), 8),
    ((1, 64, 64, 100), 4),
    ((1, 64, 64, 50), 4),      # BASELINE config 1
    ((1, 32, 32, 7), 4),
    ((3, 33, 17, 50), 4),      # partial last tile
])
def test_blob_bytes_cover_tile_blobs_and_fallback_records(shape, tp):
    lib = _cabi.load()
    p = _cabi.PertProblem()
    p.N, p.H, p.W, p.K = shape
    want_tp, want = _expected(*shape)
    assert want_tp == tp
    assert lib.pert_blob_bytes(p) == want
    assert want % 16 == 0


def test_blob_bytes_at_config2():
    lib = _cabi.load()
    p = _cabi.PertProblem()
    p.N, p.H, p.W, p.K = 8, 256, 256, 50
    # 32 768 tiles of 16 pixels: 436-word blobs (57.1 MB), then 65 536 records of 660 words (173.0 MB)
    assert lib.pert_blob_bytes(p) == 32768 * 436 * 4 + 65536 * 660 * 4
    assert lib.pert_blob_bytes(None) == 0
