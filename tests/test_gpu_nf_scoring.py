"""Neurofinder scoring on the device (csrc/regions.cu): labelling equal to scipy.ndimage.label label for label, the
validation orientation + reflect pad bit-identical to numpy, nf_mask_metrics_device bit-identical to nf_mask_metrics,
and fit validation / predict scores equal to the host loop they replace."""
import numpy as np
import pytest
import torch
from scipy import ndimage

from deepcalcium.datasets import nf

pytestmark = pytest.mark.gpu

EIGHT = np.ones((3, 3), dtype=bool)


def _row(t, kind=None):
    kind = kind if kind is not None else {torch.uint8: 0, torch.bool: 0, torch.float32: 1, torch.float64: 2}[t.dtype]
    return [t.data_ptr(), t.shape[0], t.shape[1], t.stride(0), t.stride(1), kind, 0, 0]


def _label_dev(rows, shapes):
    """dcb_label_regions over a table -> [(labels [H, W], count)]"""
    from deepcalcium.engine import ops
    h = np.asarray(rows, dtype=np.int64)
    nbytes, _ = ops.nf_score_workspace_bytes(h)
    ws = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    total = sum(H * W for H, W in shapes)
    labels = torch.full((max(total, 1),), -7, dtype=torch.int32, device='cuda')
    base = torch.empty(len(rows) + 1, dtype=torch.int32, device='cuda')
    ops.label_regions(torch.from_numpy(h).cuda(), h, labels, base, ws)
    lab, b = labels.cpu().numpy(), base.cpu().numpy()
    out, off = [], 0
    for i, (H, W) in enumerate(shapes):
        out.append((lab[off:off + H * W].reshape(H, W), int(b[i + 1] - b[i])))
        off += H * W
    return out


def _check_labels(masks):
    ts = [torch.from_numpy(np.ascontiguousarray(m, dtype=np.uint8)).cuda() for m in masks]
    got = _label_dev([_row(t) for t in ts], [m.shape for m in masks])
    for m, (lab, n) in zip(masks, got):
        ref, nref = ndimage.label(m != 0, structure=EIGHT)
        assert n == nref, (m.shape, n, nref)
        assert np.array_equal(lab, ref), m.shape


def _serpentine(H, W):
    m = np.zeros((H, W), np.uint8)
    m[::2] = 1
    for r in range(1, H, 2):
        m[r, W - 1 if (r // 2) % 2 == 0 else 0] = 1
    return m


def _spiral(n):
    m = np.zeros((n, n), np.uint8)
    top, left, bottom, right = 0, 0, n - 1, n - 1
    while top <= bottom and left <= right:
        m[top, left:right + 1] = 1
        m[top:bottom + 1, right] = 1
        if top + 2 <= bottom:
            m[bottom, left:right + 1] = 1
        if left + 2 <= right and top + 2 <= bottom:
            m[top + 2:bottom + 1, left] = 1
        top, left, bottom, right = top + 2, left + 2, bottom - 2, right - 2
        if top <= bottom and left - 1 >= 0:
            m[top, left - 1] = 1
    return m


def test_label_adversarial_shapes(cuda):
    ii, jj = np.meshgrid(np.arange(300), np.arange(301), indexing='ij')
    masks = [_serpentine(515, 477), _serpentine(64, 64), _spiral(257), _spiral(1024),
             ((ii + jj) % 2).astype(np.uint8),                      # checkerboard: one component under 8-connectivity
             ((ii + jj) % 3 == 0).astype(np.uint8),                 # anti-diagonals: joined only through up-right steps
             ((ii - jj) % 3 == 0).astype(np.uint8),
             np.ones((97, 130), np.uint8), np.zeros((97, 130), np.uint8), np.ones((1, 1), np.uint8),
             np.zeros((1, 1), np.uint8), (np.arange(1000) % 3 != 0).astype(np.uint8)[None],
             (np.arange(1000) % 3 != 0).astype(np.uint8)[:, None], np.ones((1, 700), np.uint8), np.ones((700, 1), np.uint8)]
    rng = np.random.default_rng(0)
    for shp in ((33, 31), (63, 65), (32, 32), (31, 1025)):      # around the 32 x 32 tile and the 1024-pixel chunk
        masks.append((rng.random(shp) < 0.6).astype(np.uint8))
    assert ndimage.label(masks[2], structure=EIGHT)[1] == 1 and ndimage.label(masks[3], structure=EIGHT)[1] == 1
    _check_labels(masks)                                         # one call over all of them
    for m in masks[:4]:
        _check_labels([m])


@pytest.mark.parametrize('shape', [(1, 1), (1, 511), (127, 511), (513, 67), (512, 512), (4096, 4096)])
def test_label_random_densities(cuda, shape):
    rng = np.random.default_rng(shape[0] * 7919 + shape[1])
    dens = (0.1, 0.3, 0.5, 0.6, 0.7, 0.9) if shape != (4096, 4096) else (0.1, 0.5, 0.9)
    _check_labels([(rng.random(shape) < d).astype(np.uint8) for d in dens])


def test_label_views_and_float_kinds(cuda):
    rng = np.random.default_rng(3)
    p = rng.random((130, 70)).astype(np.float32)
    p[5, 5] = np.nan
    p[7, 9] = 0.5                                  # rounds to 0
    p[9, 9] = np.nextafter(np.float32(0.5), np.float32(1))
    pd = torch.from_numpy(p).cuda()
    p64 = torch.from_numpy(p.astype(np.float64)).cuda()
    m = torch.from_numpy((rng.random((130, 70)) < 0.5).astype(np.uint8)).cuda()
    H, W = m.shape
    # np.rot90(m, 1)[a, b] = m[b, W - 1 - a]: a signed-stride view; and a crop of the float map
    rot = [m.data_ptr() + (W - 1), W, H, -1, W, 0, 0, 0]
    crop = pd[10:90, 3:61]
    rows = [rot, _row(pd), _row(p64), _row(crop)]
    got = _label_dev(rows, [(W, H), (H, W), (H, W), (80, 58)])
    refs = [np.rot90(m.cpu().numpy(), 1) != 0, np.round(p) != 0, np.round(p.astype(np.float64)) != 0,
            np.round(p[10:90, 3:61]) != 0]
    for (lab, n), ref in zip(got, refs):
        r, nr = ndimage.label(ref, structure=EIGHT)
        assert n == nr and np.array_equal(lab, r)


@pytest.mark.parametrize('hs,ws,H,W', [(512, 512, 512, 512), (300, 200, 512, 512), (600, 560, 600, 600),
                                       (384, 511, 512, 512), (3, 100, 512, 512), (1, 5, 40, 40), (7, 1, 512, 512)])
def test_orient_pad_is_numpy(cuda, hs, ws, H, W):
    from deepcalcium.engine import ops
    s = np.random.default_rng(hs * 31 + ws).standard_normal((hs, ws)).astype(np.float32)
    sd = torch.from_numpy(s).cuda()
    fwd = [lambda x: x, np.fliplr, np.flipud, lambda x: np.rot90(x, 1), lambda x: np.rot90(x, 2),
           lambda x: np.rot90(x, 3)]
    for k, f in enumerate(fwd):
        fs = f(s)
        if fs.shape[0] > H or fs.shape[1] > W:
            continue
        ref = np.pad(fs, ((0, H - fs.shape[0]), (0, W - fs.shape[1])), 'reflect')
        out = torch.full((H, W), np.nan, dtype=torch.float32, device='cuda')
        ops.orient_pad(sd, k, out)
        assert np.array_equal(out.cpu().numpy().view(np.uint32), ref.view(np.uint32)), k


# ------------------------------------------------------------------------------------------------- scoring
def _disks(rng, shape, n, rmin=2, rmax=6):
    H, W = shape
    m = np.zeros(shape, np.uint8)
    for _ in range(n):
        cy, cx, r = (int(v) for v in (rng.integers(0, H), rng.integers(0, W), rng.integers(rmin, rmax + 1)))
        y0, x0 = max(cy - r, 0), max(cx - r, 0)
        yy, xx = np.mgrid[y0:min(cy + r + 1, H), x0:min(cx + r + 1, W)]
        m[y0:y0 + yy.shape[0], x0:x0 + yy.shape[1]] |= ((yy - cy) ** 2 + (xx - cx) ** 2 <= r * r).astype(np.uint8)
    return m


def _perturb(rng, m):
    """shifted copy with dropped and merged regions and a few stray pixels"""
    lab, n = ndimage.label(m, structure=EIGHT)
    keep = rng.random(n + 1) < 0.8
    keep[0] = False
    p = keep[lab].astype(np.uint8)
    p = np.roll(p, tuple(int(v) for v in rng.integers(-3, 4, 2)), (0, 1))
    if rng.random() < 0.5:
        p = ndimage.binary_dilation(p, iterations=int(rng.integers(1, 3))).astype(np.uint8)   # merges neighbours
    p[rng.random(p.shape) < 0.002] = 1
    return p


def _rings(c, n, shape, shift=(0, 0)):
    """n concentric square rings (one 8-connected region each) all centred at c: every centre distance ties"""
    m = np.zeros(shape, np.uint8)
    cy, cx = c[0] + shift[0], c[1] + shift[1]
    for k in range(1, n + 1):
        r = 2 * k
        m[cy - r, cx - r:cx + r + 1] = m[cy + r, cx - r:cx + r + 1] = 1
        m[cy - r:cy + r + 1, cx - r] = m[cy - r:cy + r + 1, cx + r] = 1
    return m


def _hand_built():
    cases = []
    # tie: two prediction pixels at distance 3 on either side of the truth centre; the smaller label wins
    t = np.zeros((30, 30), np.uint8); t[9:12, 9:12] = 1
    p = np.zeros_like(t); p[10, 7] = p[10, 13] = 1
    cases.append((t, p))
    t2 = t.copy(); t2[20, 20] = 1
    p2 = p.copy(); p2[17, 20] = p2[23, 20] = 1               # a vertical tie as well
    cases.append((t2, p2))
    # centre pairs at exactly distance 5 (3-4-5 and 0-5): not matched; at 4.99...: matched
    t = np.zeros((40, 40), np.uint8); t[5, 5] = t[20, 5] = 1; t[30, 30] = 1
    p = np.zeros_like(t); p[8, 9] = p[20, 10] = 1; p[33, 33] = 1
    cases.append((t, p))
    # many-to-one: two truth regions compete for one prediction region; the first in label order takes it
    t = np.zeros((20, 60), np.uint8); t[10, 30] = t[10, 36] = t[10, 50] = 1
    p = np.zeros_like(t); p[10, 33] = p[10, 52] = 1
    cases.append((t, p))
    # eight nested rings against eight nested rings: every distance ties, more candidates than the kept list
    cases.append((_rings((40, 40), 8, (81, 81)), _rings((40, 40), 8, (81, 81))))
    cases.append((_rings((40, 40), 8, (81, 81)), _rings((40, 40), 7, (81, 81), shift=(1, 0))))
    # empty truth with a prediction (recall NaN); empty prediction (zeros); both empty
    z = np.zeros((25, 17), np.uint8); q = z.copy(); q[3:6, 3:6] = 1
    cases += [(z, q), (q, z), (z, z.copy())]
    return cases


def _corpus(seed=11, n=520):
    rng = np.random.default_rng(seed)
    cases = _hand_built()
    shapes = [(128, 511), (64, 64), (37, 129), (200, 90), (1, 40), (40, 1), (512, 512)]
    while len(cases) < n:
        shp = shapes[len(cases) % len(shapes)] if rng.random() < 0.7 else tuple(int(v) for v in rng.integers(1, 160, 2))
        area = shp[0] * shp[1]
        t = _disks(rng, shp, max(1, area // 900))
        if rng.random() < 0.1:
            t = (rng.random(shp) < rng.random()).astype(np.uint8)
        cases.append((t, _perturb(rng, t)))
    return cases


def _to_device(cases, seed=5):
    """mixed dtypes and strided views of the corpus"""
    rng = np.random.default_rng(seed)
    out = []
    for i, (t, p) in enumerate(cases):
        def dev(a, j):
            k = (i + j) % 5
            if k == 0:
                return torch.from_numpy(a).cuda()
            if k == 1:
                return torch.from_numpy(a.astype(bool)).cuda()
            if k == 2:
                return torch.from_numpy(a.astype(np.float32)).cuda()
            if k == 3:
                return torch.from_numpy(a.astype(np.float64)).cuda()
            big = torch.zeros(a.shape[0] + 5, a.shape[1] + 9, dtype=torch.uint8, device='cuda')
            big[2:2 + a.shape[0], 4:4 + a.shape[1]] = torch.from_numpy(a).cuda()
            return big[2:2 + a.shape[0], 4:4 + a.shape[1]]             # a row-strided view
        out.append((dev(t, 0), dev(p, 1)))
    return out


def _eq(a, b):
    return np.array_equal(np.asarray(a, np.float64), np.asarray(b, np.float64), equal_nan=True)


def test_device_scores_equal_host_scores_bit_for_bit(cuda):
    cases = _corpus()
    assert len(cases) >= 500
    pairs = _to_device(cases)
    got = nf.nf_mask_metrics_device(pairs)
    assert len(got) == len(cases)
    nan_seen = matched = 0
    for i, ((t, p), g) in enumerate(zip(cases, got)):
        ref = nf.nf_mask_metrics(t, p)
        assert _eq(g, ref), (i, t.shape, g, ref)
        nan_seen += bool(np.isnan(ref).any())
        matched += ref[1] > 0
    assert nan_seen >= 1 and matched > 400
    # the hand-built cases score what the matching rules say
    assert got[0][:2] == (0.5, 1.0) and got[2][:2] == (1 / 3, 1 / 3) and got[3][:2] == (1.0, 2 / 3)
    assert got[4] == (1.0, 1.0, 1.0, 1.0, 1.0)
    assert got[8] == (0., 0., 0., 0., 0.) and got[7] == (0., 0., 0., 0., 0.) and np.isnan(got[6][1])


def test_batched_equals_per_pair_and_repeats(cuda):
    cases = _corpus(seed=12, n=60)
    pairs = _to_device(cases, seed=6)
    once = nf.nf_mask_metrics_device(pairs)
    again = nf.nf_mask_metrics_device(pairs)
    single = [nf.nf_mask_metrics_device([pr])[0] for pr in pairs]
    assert _eq(once, again) and _eq(once, single)
    with pytest.raises(ValueError):
        nf.nf_mask_metrics_device([(pairs[0][0], pairs[1][1][:3, :3])])
    with pytest.raises(TypeError):
        nf.nf_mask_metrics_device([(pairs[0][0].cpu(), pairs[0][1].cpu())])


def test_bad_tables_are_rejected(cuda):
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    t = torch.zeros(4, 4, dtype=torch.uint8, device='cuda')
    for bad in ([_row(t)[:5] + [3, 0, 0]], [[t.data_ptr(), -1, 4, 4, 1, 0, 0, 0]], [[0, 4, 4, 4, 1, 0, 0, 0]]):
        with pytest.raises(nat.DcbError):
            ops.nf_score_workspace_bytes(np.asarray(bad, dtype=np.int64))
    h = np.asarray([_row(t), _row(t[:3])], dtype=np.int64)
    nbytes, cap = ops.nf_score_workspace_bytes(h)
    with pytest.raises(nat.DcbError):
        ops.nf_score(torch.from_numpy(h).cuda(), h, torch.empty(3, dtype=torch.int32, device='cuda'),
                     torch.empty(cap, 3, dtype=torch.int32, device='cuda'), torch.empty(nbytes, dtype=torch.uint8, device='cuda'))


# ------------------------------------------------------------------------------------------------- integration
def _host_validate(model, S_summ, M_summ, y_coords, shape_val, epoch):
    """UNet2DSummary._validate as it ran on the host before the device path; also returns the predicted region counts"""
    hw, ww = shape_val

    def pad(x):
        return np.pad(x, ((0, hw - x.shape[0]), (0, ww - x.shape[1])), 'reflect')

    def predict(x):
        if x.shape[0] <= hw and x.shape[1] <= ww:
            return model.predict(pad(x)[np.newaxis, :, :])[0][:x.shape[0], :x.shape[1]]
        xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(model.engine.dev)
        return model.engine.predict_tiled(xd, augmentation=False)[1].cpu().numpy()

    fwd = [lambda x: x, np.fliplr, np.flipud, lambda x: np.rot90(x, 1), lambda x: np.rot90(x, 2),
           lambda x: np.rot90(x, 3)]
    pp, rr, ff, nreg = [], [], [], []
    for s, m, (y0, y1) in zip(S_summ, M_summ, y_coords):
        vm = np.zeros(s.shape, dtype=np.uint8)
        vm[y0:y1, :] = 1
        for f in fwd:
            fs, fm = f(s), f(m)
            yy, xx = np.where(f(vm) == 1)
            a0, a1, b0, b1 = min(yy), max(yy), min(xx), max(xx)
            mp = predict(fs)
            p, r, _, _, f1 = nf.nf_mask_metrics(fm[a0:a1, b0:b1], mp[a0:a1, b0:b1].round())
            nreg.append(len(nf._label_regions(mp[a0:a1, b0:b1].round())))
            pp.append(p); rr.append(r); ff.append(f1)
    eps = 1e-4 * epoch if epoch else 0
    return {'val_nf_f1_mean': float(np.mean(ff) + eps), 'val_nf_f1_median': float(np.median(ff) + eps),
            'val_nf_f1_min': float(np.min(ff) + eps), 'val_nf_f1_adj': float(np.mean(ff) * np.min(ff) + eps),
            'val_nf_prec': float(np.mean(pp)), 'val_nf_reca': float(np.mean(rr))}, nreg


def _data(seed, shapes):
    rng = np.random.default_rng(seed)
    S, M = [], []
    for shp in shapes:
        m = _disks(rng, shp, shp[0] * shp[1] // 2500, 3, 6).astype(np.float64)
        s = ndimage.gaussian_filter(rng.standard_normal(shp), 2) + 2 * ndimage.gaussian_filter(m, 1)
        S.append(((s - s.mean()) / s.std()).astype(np.float32))
        M.append(m)
    return S, M


def _many_regions(model, S, frac=0.35):
    """shift head/bias so that about `frac` of the pixels of the first image are predicted foreground: with random
    weights that gives many separate regions in every orientation"""
    w = model.engine.get_weights_dict()
    x = np.pad(S[0], ((0, 512 - S[0].shape[0]), (0, 512 - S[0].shape[1])), 'reflect')[None] if max(S[0].shape) <= 512 \
        else S[0][None, :512, :512]
    logit = model.predict_logits(x)[0]
    w['head/bias'] = w['head/bias'].copy()
    w['head/bias'][1] -= np.quantile(logit, 1 - frac)
    model.engine.set_weights_dict(w)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_validate_on_device_equals_host_loop(cuda, precision):
    from deepcalcium.models.neurons import UNet2DSummary, unet
    S, M = _data(21, [(512, 512), (300, 420), (600, 560)])
    y_coords = [(s.shape[0] - int(s.shape[0] * 0.25), s.shape[0]) for s in S]
    model = unet((128, 128), nb_filters_base=8, precision=precision, seed=4)
    _many_regions(model, S)
    api = UNet2DSummary.__new__(UNet2DSummary)
    for epoch in (0, 3):
        host, nreg = _host_validate(model, S, M, y_coords, (512, 512), epoch)
        dev = api._validate(model, S, M, None, y_coords, (512, 512), epoch)
        assert min(nreg) >= 10, nreg
        assert dev.keys() == host.keys()
        for k in host:
            assert _eq(dev[k], host[k]), (k, dev[k], host[k])


def test_predict_scores_equal_host_scoring(cuda, tmp_path):
    from deepcalcium.models.neurons import UNet2DSummary, unet
    S, M = _data(22, [(512, 512), (400, 500), (600, 560)])
    model = unet((512, 512), nb_filters_base=8, precision='bf16', seed=5)
    _many_regions(model, S, 0.3)
    names = ['a', 'b', 'c']
    api = UNet2DSummary(cpdir=str(tmp_path / 'cp'), dataset_name_func=lambda p: p,
                        series_summary_func=lambda p: S[names.index(p)], mask_summary_func=lambda p: M[names.index(p)])
    for aug in (False, True):
        Mp, _ = api.predict(names, model, print_scores=True, augmentation=aug)
        scores = [0., 0., 0.]
        for m, mp in zip(M, Mp):
            p, r, _, _, comb = nf.nf_mask_metrics(m, mp.round())
            for k, v in enumerate((p, r, comb)):
                scores[k] += v / len(names)
        assert len(nf._label_regions(Mp[0])) >= 10
        assert _eq([api.last_scores[k] for k in ('prec', 'reca', 'comb')], scores), (api.last_scores, scores)
