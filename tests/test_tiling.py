"""Overlap-tile inference for summary images larger than the 512^2 window, on the CPU: the tile planner's invariants, the
network's receptive reach (structural pass over the graph, checked on the oracle), and the stitching arithmetic of
dcb_tile_make_batch / dcb_tile_combine (their numpy statements) against whole-canvas TTA in the oracle."""
import numpy as np
import pytest
import torch

import oracle
from deepcalcium.engine.graph import GraphSpec, MAX_TILE, plan_tiles, receptive_reach, tile_halo
from deepcalcium.utils.neurons import INVERTIBLE_2D_AUGMENTATIONS, tile_combine_host, tile_make_batch_host

HALO = 96


def _owner_counts_and_margins(plan):
    """per canvas pixel, along each dimension: how many tiles own it, and its least distance to an owning tile's edge
    that is not a canvas edge"""
    out = []
    for d in (0, 1):
        C, T = plan.canvas[d], plan.tile
        o, c = plan.origins[d], plan.cuts[d]
        count = np.zeros(C, int)
        margin = np.full(C, np.iinfo(int).max)
        for k, ok in enumerate(o):
            lo = c[k - 1] if k > 0 else 0
            hi = c[k] if k < len(o) - 1 else C
            count[lo:hi] += 1
            px = np.arange(lo, hi)
            if ok > 0:
                margin[lo:hi] = np.minimum(margin[lo:hi], px - ok)
            if ok + T < C:
                margin[lo:hi] = np.minimum(margin[lo:hi], ok + T - 1 - px)
        out.append((count, margin))
    return out


@pytest.mark.parametrize('tile', [224, 512, 640, 1024, None])
@pytest.mark.parametrize('shape', [(1, 1), (100, 1100), (300, 250), (512, 512), (513, 512), (700, 530), (796, 512),
                                   (1040, 600), (1300, 900), (2048, 2048), (4096, 4096), (5000, 3001)])
def test_plan_owns_every_canvas_pixel_once_away_from_inner_tile_edges(shape, tile):
    plan = plan_tiles(shape, HALO, tile)
    T = plan.tile
    assert T % 16 == 0 and T > 2 * HALO
    if tile is None:
        assert T % 128 == 0 and 512 <= T <= MAX_TILE
    for d in (0, 1):
        C = plan.canvas[d]
        assert C == max(T, -(-shape[d] // 16) * 16)
        assert all(o % 16 == 0 and 0 <= o <= C - T for o in plan.origins[d])
        assert plan.origins[d] == sorted(plan.origins[d]) and plan.origins[d][0] == 0
    for count, margin in _owner_counts_and_margins(plan):
        assert np.all(count == 1)
        assert np.all(margin >= HALO)


@pytest.mark.parametrize('shape', [(1, 1), (200, 512), (500, 480), (512, 512)])
def test_images_of_at_most_512_get_one_512_tile(shape):
    plan = plan_tiles(shape, HALO)
    assert plan.tile == 512 and plan.canvas == (512, 512) and plan.n_tiles == 1


def test_automatic_tile_minimises_computed_pixels():
    for shape in [(796, 512), (1024, 1024), (1300, 900), (4096, 4096)]:
        plan = plan_tiles(shape, HALO)
        for T in range(512, MAX_TILE + 1, 128):
            assert plan.computed_pixels() <= plan_tiles(shape, HALO, T).computed_pixels()
    assert plan_tiles((2048, 2048), HALO).n_tiles == 1
    with pytest.raises(ValueError):
        plan_tiles((600, 600), HALO, tile=200)              # not a multiple of 16
    with pytest.raises(ValueError):
        plan_tiles((600, 600), HALO, tile=192)              # no room for an owned pixel


@pytest.mark.parametrize('mode', ['transpose', 'upsampling'])
def test_structural_receptive_reach_is_94(mode):
    for nfb in (4, 32):
        spec = GraphSpec(nfb, upsampling_or_transpose=mode)
        assert receptive_reach(spec) == (94, 94)
        assert tile_halo(spec) == HALO


def test_oracle_dependency_of_a_16_block_matches_the_reach():
    """outputs 160..175 (rows and columns) of a 352^2 forward depend on input rows / columns 66..269 and no others:
    replacing every input pixel outside that square leaves them unchanged, changing row or column 66 or 269 does not"""
    spec = oracle.UNetSpec(4)
    rng = np.random.default_rng(0)
    x = rng.standard_normal((1, 352, 352))
    blk = (slice(None), slice(160, 176), slice(160, 176))
    lo, hi = 160 - 94, 175 + 94
    for seed in (1, 2, 3):
        w = oracle.init_weights(spec, seed=seed)

        def fwd(a):
            with torch.no_grad():
                return oracle.unet_forward(w, a, spec, dtype=torch.float64)['logit'].numpy()[blk]

        base = fwd(x)
        far = rng.standard_normal(x.shape)
        far[:, lo:hi + 1, lo:hi + 1] = x[:, lo:hi + 1, lo:hi + 1]
        assert np.max(np.abs(fwd(far) - base)) < 1e-12
        for edge in (lo, hi):
            for axis in (1, 2):
                x2 = x.copy()
                idx = [slice(None)] * 3
                idx[axis] = edge
                x2[tuple(idx)] += 10.0
                assert np.max(np.abs(fwd(x2) - base)) > 1e-9, (seed, edge, axis)


def test_stitched_tiles_equal_whole_canvas_tta_in_the_oracle():
    """nfb 4, float64, a 300 x 250 image with 224^2 tiles (4 x 2 of them): per-tile 8x TTA cut by the numpy statement of
    dcb_tile_make_batch and stitched by the one of dcb_tile_combine equals the TTA of the whole canvas.  Both sides sum
    p / 8 in float64 (no float32 rounding), so last-bit differences in p cannot flip a rounding."""
    spec = oracle.UNetSpec(4)
    w = oracle.init_weights(spec, seed=11)
    s = np.random.default_rng(12).standard_normal((300, 250)).astype(np.float32)
    plan = plan_tiles(s.shape, HALO, tile=224)
    assert plan.grid == (4, 2) and plan.canvas == (304, 256)

    def forward(xb):
        with torch.no_grad():
            return oracle.unet_forward(w, np.ascontiguousarray(xb), spec, dtype=torch.float64)['prob'].numpy()

    (oy, ox), (cy, cx) = plan.origins, plan.cuts
    batch = tile_make_batch_host(s, plan.tile, oy, ox, 0, plan.n_tiles, 0, 8)
    tiled = tile_combine_host(forward(batch), plan.tile, 300, 250, oy, ox, cy, cx, 0, plan.n_tiles, 8)
    # the same stitching, one tile per group, in reverse order: every pixel is written once
    regrouped = np.full((300, 250), np.nan)
    for t in reversed(range(plan.n_tiles)):
        tile_combine_host(forward(batch[8 * t:8 * t + 8]), plan.tile, 300, 250, oy, ox, cy, cx, t, 1, 8, act=regrouped)
    assert np.array_equal(regrouped, tiled)

    canvas = np.pad(s.astype(np.float64), ((0, 4), (0, 6)), mode='reflect')[None]
    whole = np.zeros((300, 250))
    for _, aug, inv in INVERTIBLE_2D_AUGMENTATIONS:
        whole += inv(forward(aug(canvas)))[0, :300, :250] / 8
    assert np.max(np.abs(tiled - whole)) < 1e-12


def test_host_batch_of_the_one_tile_plan_is_the_reflect_padded_window():
    s = np.random.default_rng(3).standard_normal((27, 30)).astype(np.float32)
    out = tile_make_batch_host(s, 32, [0], [0], 0, 1, 0, 8)
    padded = oracle.reflect_pad(s, 32, 32)[None]
    for k, (name, aug, _) in enumerate(INVERTIBLE_2D_AUGMENTATIONS):
        assert np.array_equal(out[k], aug(padded)[0]), name
