"""Overlap-tile inference on the GPU for summary images larger than the 512^2 window: dcb_tile_make_batch /
dcb_tile_combine against their numpy statements, UNetEngine.predict_tiled against whole-canvas TTA (fp32 check mode and
fp16), against predict_tta for images that fit the window, across group sizes and graph replays, and through the
UNet2DSummary predict / fit surface."""
import numpy as np
import pytest
import torch

import oracle
from deepcalcium.engine.graph import plan_tiles
from deepcalcium.utils.neurons import INVERTIBLE_2D_AUGMENTATIONS, tile_combine_host, tile_make_batch_host

pytestmark = pytest.mark.gpu


def _engine(nfb, precision, seed=7535):
    from deepcalcium.engine.graph import GraphSpec
    from deepcalcium.engine.unet_engine import UNetEngine
    eng = UNetEngine(GraphSpec(nfb), precision=precision)
    eng.set_weights_dict(oracle.init_weights(oracle.UNetSpec(nfb), seed=seed))
    return eng


def _i32(v):
    return torch.tensor(v, dtype=torch.int32, device='cuda')


def _groups(n, size):
    return [(t0, min(size, n - t0)) for t0 in range(0, n, size)]


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize('shape,tile', [((300, 250), 224), ((250, 300), 224), ((37, 61), 224), ((1000, 37), 256)])
def test_tile_make_batch_matches_the_host_statement(cuda, dtype, shape, tile):
    from deepcalcium.engine import ops
    s = np.random.default_rng(1).standard_normal(shape).astype(np.float32)
    plan = plan_tiles(shape, 96, tile)
    (oy, ox), n = plan.origins, plan.n_tiles
    sd = torch.from_numpy(s).cuda()
    for first, count in ((0, 8), (0, 1), (3, 4)):
        for size in sorted({1, 3, n}):
            for t0, nt in _groups(n, size):
                out = torch.empty(nt * count, tile, tile, dtype=dtype, device='cuda')
                ops.tile_make_batch(sd, tile, _i32(oy), _i32(ox), t0, nt, first, count, out)
                ref = torch.from_numpy(tile_make_batch_host(s, tile, oy, ox, t0, nt, first, count)).to(dtype)
                assert torch.equal(out.cpu(), ref), (first, count, t0, nt)


@pytest.mark.parametrize('n_aug', [1, 8])
@pytest.mark.parametrize('shape,tile', [((300, 250), 224), ((250, 300), 224), ((37, 61), 224), ((1000, 37), 256)])
def test_tile_combine_matches_the_host_statement_for_every_grouping(cuda, n_aug, shape, tile):
    from deepcalcium.engine import ops
    hs, ws = shape
    plan = plan_tiles(shape, 96, tile)
    (oy, ox), (cy, cx), n = plan.origins, plan.cuts, plan.n_tiles
    probs = np.random.default_rng(2).random((n * n_aug, tile, tile)).astype(np.float32)
    ref = tile_combine_host(probs, tile, hs, ws, oy, ox, cy, cx, 0, n, n_aug)
    dp = torch.from_numpy(probs).cuda()
    for size in sorted({1, 3, n}):
        act = torch.full((hs, ws), float('nan'), dtype=torch.float64, device='cuda')
        mask = torch.full((hs, ws), 7, dtype=torch.uint8, device='cuda')
        for t0, nt in _groups(n, size):
            ops.tile_combine(dp[t0 * n_aug:(t0 + nt) * n_aug], tile, _i32(oy), _i32(ox), _i32(cy), _i32(cx), t0, nt, 0.5,
                             n_aug, act, mask)
        assert np.array_equal(act.cpu().numpy(), ref), size           # also: no pixel left unwritten (NaN)
        assert np.array_equal(mask.cpu().numpy(), (ref > 0.5).astype(np.uint8)), size


@pytest.mark.parametrize('shape', [(500, 480), (512, 512)])
@pytest.mark.parametrize('augmentation', [True, False])
def test_one_tile_plan_is_bit_identical_to_predict_tta(cuda, shape, augmentation):
    eng = _engine(32, 'fp16')
    s = torch.from_numpy(np.random.default_rng(3).standard_normal(shape).astype(np.float32)).cuda()
    m0, a0 = (t.clone() for t in eng.predict_tta(s, augmentation=augmentation))
    for _ in range(3):                                   # eager, capture + replay, replay
        m1, a1 = eng.predict_tiled(s, augmentation=augmentation, tile=512)
        assert torch.equal(m1, m0) and torch.equal(a1, a0)
    m2, a2 = eng.predict_tiled(s, augmentation=augmentation)          # the planner's choice for <= 512 is that plan
    assert torch.equal(m2, m0) and torch.equal(a2, a0)


def _whole_canvas_tta(eng, s, canvas, augmentation=True):
    """the reference's TTA with the window = the canvas (engine.infer on each transformed canvas): act float64 [hs, ws]"""
    hs, ws = s.shape
    c = np.pad(s, ((0, canvas[0] - hs), (0, canvas[1] - ws)), mode='reflect')[None]
    table = INVERTIBLE_2D_AUGMENTATIONS if augmentation else INVERTIBLE_2D_AUGMENTATIONS[:1]
    act = np.zeros((hs, ws))
    for _, aug, inv in table:
        prob, _ = eng.infer(torch.from_numpy(np.ascontiguousarray(aug(c))).cuda())
        act += inv(prob.cpu().numpy())[0, :hs, :ws] / np.float32(len(table))
    return act


@pytest.mark.parametrize('nfb', [4, 32])
@pytest.mark.parametrize('shape', [(700, 530), (1040, 600)])
def test_tiled_equals_whole_canvas_tta_fp32(cuda, nfb, shape):
    eng = _engine(nfb, 'fp32')
    s = np.random.default_rng(4).standard_normal(shape).astype(np.float32)
    plan = plan_tiles(shape, eng.halo, 512)
    assert plan.n_tiles >= 2
    ref = _whole_canvas_tta(eng, s, plan.canvas)
    mask, act = eng.predict_tiled(torch.from_numpy(s).cuda(), tile=512)
    act, mask = act.cpu().numpy(), mask.cpu().numpy()
    assert np.max(np.abs(act - ref)) < 1e-5
    flips = mask != (ref > 0.5)
    assert np.all(np.abs(ref[flips] - 0.5) < 1e-5)


@pytest.mark.parametrize('shape', [(1024, 1024), (1300, 900)])
def test_tiled_fp16_against_the_whole_canvas(cuda, shape):
    """north-star tolerances: act within 1e-2, masks differ on at most 0.1 % of pixels.  The 1024^2 canvas is the same for
    512^2 tiles and for one 1024^2 tile; the 1312 x 912 canvas of the 512^2 plan fits no square tile, so there the
    reference is the whole-canvas TTA run through engine.infer."""
    eng = _engine(32, 'fp16')
    s = np.random.default_rng(5).standard_normal(shape).astype(np.float32)
    sd = torch.from_numpy(s).cuda()
    plan = plan_tiles(shape, eng.halo, 512)
    if shape[0] == shape[1]:
        _, a1 = eng.predict_tiled(sd, tile=shape[0])
        ref = a1.cpu().numpy()
    else:
        ref = _whole_canvas_tta(eng, s, plan.canvas)
    mask, act = eng.predict_tiled(sd, tile=512)
    err = float(np.max(np.abs(act.cpu().numpy() - ref)))
    dis = float(np.mean(mask.cpu().numpy() != (ref > 0.5)))
    print('tiled fp16 %s (%d tiles of 512^2): max |act diff| %.3g, mask disagreement %.5f' % (shape, plan.n_tiles, err, dis))
    assert err < 1e-2 and dis <= 1e-3


def test_tiled_results_are_bit_identical_across_graph_replays_and_close_across_groupings(cuda):
    """for each group size: the eager call, the capture and a replay agree bit for bit.  Across group sizes the stitching
    is exact (tile_combine writes each pixel once, see the kernel test above), but the forward runs on a batch of a
    different size, for which the convolution kernels may pick a different work split: equal up to float rounding."""
    eng = _engine(32, 'fp16')
    s = torch.from_numpy(np.random.default_rng(6).standard_normal((1040, 600)).astype(np.float32)).cuda()
    assert plan_tiles(s.shape, eng.halo, 512).n_tiles == 6
    first = {}
    for per_group in (1, 4, 6):                          # 4: a group of 4 tiles and a last group of 2
        eng.tile_batch_pixels = per_group * 8 * 512 * 512
        runs = [tuple(t.clone() for t in eng.predict_tiled(s, tile=512)) for _ in range(3)]   # eager, capture, replay
        for m, a in runs[1:]:
            assert torch.equal(m, runs[0][0]) and torch.equal(a, runs[0][1]), per_group
        first[per_group] = runs[0]
    for per_group, (m, a) in first.items():
        err = float((a - first[1][1]).abs().max())
        dis = float((m != first[1][0]).double().mean())
        print('group of %d tiles vs 1: max |act diff| %.3g, mask disagreement %.6f' % (per_group, err, dis))
        assert err < 1e-3 and dis <= 1e-4


def test_summary_predict_mixes_window_and_tiled_images(cuda, tmp_path):
    from deepcalcium.models.neurons import UNet2DSummary
    from deepcalcium.models.neurons.unet_2d_summary import UNetModel
    from deepcalcium.engine.graph import GraphSpec
    eng = _engine(32, 'fp16')
    rng = np.random.default_rng(7)
    shapes = [(500, 480), (900, 700), (512, 512), (1100, 1100), (900, 700), (500, 480)]
    imgs = {('img%d' % i): rng.standard_normal(shp).astype(np.float32) for i, shp in enumerate(shapes)}
    model = UNetModel.__new__(UNetModel)
    model.window_shape, model.spec, model.engine = (512, 512), GraphSpec(32), eng
    api = UNet2DSummary(cpdir=str(tmp_path / 'cp'), dataset_name_func=lambda p: p, series_summary_func=lambda p: imgs[p])
    paths = list(imgs.keys())
    for aug in (True, False):
        first = None
        for rep in range(2):
            Mp, names = api.predict(paths, model, augmentation=aug)
            assert names == paths
            for p_, mp in zip(paths, Mp):
                sd = torch.from_numpy(imgs[p_]).cuda()
                if max(imgs[p_].shape) <= 512:
                    ref = eng.predict_tta(sd, augmentation=aug)[0]
                else:
                    ref = eng.predict_tiled(sd, augmentation=aug)[0]
                assert mp.shape == imgs[p_].shape and np.array_equal(mp, ref.cpu().numpy()), (aug, rep, p_)
            if first is None:
                first = Mp
            assert all(np.array_equal(a, b) for a, b in zip(first, Mp))


def test_fit_validates_an_image_larger_than_the_validation_window(cuda, tmp_path):
    from deepcalcium.models.neurons import UNet2DSummary, unet
    from deepcalcium.models.neurons.unet_2d_summary import Adam
    from deepcalcium.datasets.nf import make_dataset
    rng = np.random.default_rng(8)
    masks = np.zeros((20, 600, 560), np.int8)
    for k in range(20):
        cy, cx = rng.integers(10, 590), rng.integers(10, 550)
        masks[k, cy - 4:cy + 4, cx - 4:cx + 4] = 1
    movie = rng.random((20, 600, 560)).astype(np.float32) * 50 + masks.max(0)[None] * 100 * rng.random((20, 1, 1))
    path = make_dataset(str(tmp_path / 'big.npz'), 'synthetic.big', movie=movie.astype(np.float32), masks=masks)
    np.random.seed(865)
    model = UNet2DSummary(cpdir=str(tmp_path / 'cp'),
                          net_builder_func=lambda shape: unet(shape, nb_filters_base=32, precision='bf16'))
    hist, _ = model.fit([path], shape_trn=(64, 64), shape_val=(512, 512), batch_size_trn=4, nb_steps_trn=2, nb_epochs=1,
                        optimizer=Adam(0.002), loss='dice_loss')
    # a network trained for two steps may match no neuron in an orientation, and then the neurofinder F1 is 0 / 0 = NaN
    # (as in the reference); precision and recall are always defined
    assert len(hist['val_nf_f1_mean']) == 1
    assert np.isfinite(hist['val_nf_prec'][0]) and np.isfinite(hist['val_nf_reca'][0])
