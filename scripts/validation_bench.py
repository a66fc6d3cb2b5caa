"""What fit validation and Neurofinder scoring cost on the host and on the device.

    python scripts/validation_bench.py [--out profiles/validation_b200.json] [--skip-fit]

(a) Scoring only: 114 seeded (truth, prediction) pairs - 19 datasets x 6 orientations of 128 x 511 validation crops with
    about 75 disk neurons each; the predictions are the truth shifted, with regions dropped and neighbours merged.  The
    host loop of nf_mask_metrics against one nf_mask_metrics_device call (including its device-to-host copies).
(b) UNet2DSummary._validate end to end at nb_filters_base 32, bf16, on 19 synthetic 512^2 datasets with 300 disk neurons
    each (the size of the Neurofinder training set): host_validate below (the host loop _validate ran before it moved to
    the device) against the device path.  head/bias is shifted so that about 10 % of each window is predicted foreground,
    so the scoring sees realistic region counts; the counts are reported.
(c) One fit epoch at the CLI's configuration (examples/neurons/unet2ds_nf.py: 100 steps of 20 crops of 128^2, 512^2
    validation) on the same 19 datasets (given as arrays, so no dataset files and no _summarize_mask), with _validate as
    it is and with host_validate patched in.
Both paths must give the same numbers; the script checks that.  The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'deep-calcium_b200')); sys.path.insert(0, ROOT)
os.environ.setdefault('DEEP_CALCIUM_HOME', os.path.join(tempfile.gettempdir(), 'deep-calcium-home'))
sys.path.insert(0, os.path.join(ROOT, 'scripts'))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy import ndimage  # noqa: E402
from deepcalcium.datasets import nf  # noqa: E402
from deepcalcium.models.neurons import UNet2DSummary, unet  # noqa: E402
from large_image_bench import gpu_info  # noqa: E402

EIGHT = np.ones((3, 3), bool)
FWD = [lambda x: x, np.fliplr, np.flipud, lambda x: np.rot90(x, 1), lambda x: np.rot90(x, 2), lambda x: np.rot90(x, 3)]


def disks(rng, shape, n, rmin=4, rmax=7):
    H, W = shape
    m = np.zeros(shape, np.uint8)
    for _ in range(n):
        cy, cx, r = (int(v) for v in (rng.integers(0, H), rng.integers(0, W), rng.integers(rmin, rmax + 1)))
        y0, x0 = max(cy - r, 0), max(cx - r, 0)
        yy, xx = np.mgrid[y0:min(cy + r + 1, H), x0:min(cx + r + 1, W)]
        m[y0:y0 + yy.shape[0], x0:x0 + yy.shape[1]] |= ((yy - cy) ** 2 + (xx - cx) ** 2 <= r * r).astype(np.uint8)
    return m


def perturb(rng, m):
    lab, n = ndimage.label(m, structure=EIGHT)
    keep = rng.random(n + 1) < 0.85
    keep[0] = False
    p = np.roll(keep[lab].astype(np.uint8), tuple(int(v) for v in rng.integers(-2, 3, 2)), (0, 1))
    if rng.random() < 0.3:
        p = ndimage.binary_dilation(p).astype(np.uint8)
    return p


def host_validate(model, S_summ, M_summ, y_coords, shape_val, epoch):
    """UNet2DSummary._validate as it ran on the host: numpy orientation + reflect pad, batch-1 forward, download,
    np.where box, nf_mask_metrics.  Also returns the predicted region count of every crop."""
    hw, ww = shape_val
    pp, rr, ff, nreg = [], [], [], []
    for s, m, (y0, y1) in zip(S_summ, M_summ, y_coords):
        vm = np.zeros(s.shape, dtype=np.uint8)
        vm[y0:y1, :] = 1
        for f in FWD:
            fs, fm = f(s), f(m)
            yy, xx = np.where(f(vm) == 1)
            a0, a1, b0, b1 = min(yy), max(yy), min(xx), max(xx)
            if fs.shape[0] <= hw and fs.shape[1] <= ww:
                x = np.pad(fs, ((0, hw - fs.shape[0]), (0, ww - fs.shape[1])), 'reflect')
                mp = model.predict(x[np.newaxis])[0][:fs.shape[0], :fs.shape[1]]
            else:
                xd = torch.from_numpy(np.ascontiguousarray(fs, dtype=np.float32)).to(model.engine.dev)
                mp = model.engine.predict_tiled(xd, augmentation=False)[1].cpu().numpy()
            p, r, _, _, f1 = nf.nf_mask_metrics(fm[a0:a1, b0:b1], mp[a0:a1, b0:b1].round())
            nreg.append(int(ndimage.label(mp[a0:a1, b0:b1].round() != 0, structure=EIGHT)[1]))
            pp.append(p); rr.append(r); ff.append(f1)
    eps = 1e-4 * epoch if epoch else 0
    logs = {'val_nf_f1_mean': float(np.mean(ff) + eps), 'val_nf_f1_median': float(np.median(ff) + eps),
            'val_nf_f1_min': float(np.min(ff) + eps), 'val_nf_f1_adj': float(np.mean(ff) * np.min(ff) + eps),
            'val_nf_prec': float(np.mean(pp)), 'val_nf_reca': float(np.mean(rr))}
    return logs, nreg


def same(a, b):
    return np.array_equal(np.asarray(a, np.float64), np.asarray(b, np.float64), equal_nan=True)


def wall(fn, reps):
    torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        t.append(time.perf_counter() - t0)
    return out, float(np.median(t)), t


def bench_scoring(rng):
    cases = []
    for _ in range(19):
        full = disks(rng, (512, 512), 300)
        for f in FWD:
            t = np.ascontiguousarray(f(full)[384:512, 0:511])
            cases.append((t, perturb(rng, t)))
    host, t_host, _ = wall(lambda: [nf.nf_mask_metrics(t, p) for t, p in cases], 2)
    dev_pairs = [(torch.from_numpy(t).cuda(), torch.from_numpy(p).cuda()) for t, p in cases]
    nf.nf_mask_metrics_device(dev_pairs)
    dev, t_dev, ts = wall(lambda: nf.nf_mask_metrics_device(dev_pairs), 20)
    assert all(same(a, b) for a, b in zip(host, dev)), 'device scores differ from the host'
    na = [len(nf._label_regions(t)) for t, _ in cases]
    return {'pairs': len(cases), 'crop': [128, 511], 'truth_regions_mean': float(np.mean(na)),
            'host_s': t_host, 'device_s': t_dev, 'device_s_all': ts, 'speedup': t_host / t_dev, 'bit_identical': True}


def make_data(rng, n=19):
    S, M = [], []
    for _ in range(n):
        m = disks(rng, (512, 512), 300).astype(np.float64)
        s = ndimage.gaussian_filter(rng.standard_normal((512, 512)), 2) + 3 * ndimage.gaussian_filter(m, 1.5)
        S.append(((s - s.mean()) / s.std()).astype(np.float32))
        M.append(m)
    return S, M


def shift_head(model, S, frac=0.10):
    w = model.engine.get_weights_dict()
    logit = model.predict_logits(S[0][None])[0]
    w['head/bias'] = w['head/bias'].copy()
    w['head/bias'][1] -= np.quantile(logit, 1 - frac)
    model.engine.set_weights_dict(w)


def bench_validate(S, M):
    model = unet((128, 128), nb_filters_base=32, precision='bf16', seed=3)
    shift_head(model, S)
    y_coords = [(s.shape[0] - int(s.shape[0] * 0.25), s.shape[0]) for s in S]
    api = UNet2DSummary.__new__(UNet2DSummary)
    val = api._validation_data(S, M, model.engine.dev)
    (host, nreg), t_host, _ = wall(lambda: host_validate(model, S, M, y_coords, (512, 512), 1), 2)
    api._validate(model, S, M, None, y_coords, (512, 512), 1, val)
    dev, t_dev, ts = wall(lambda: api._validate(model, S, M, None, y_coords, (512, 512), 1, val), 5)
    assert all(same(dev[k], host[k]) for k in host), (dev, host)
    # the 114 batch-1 forwards alone, for the share of the device path that is network time
    win = torch.from_numpy(S[0]).cuda()[None]
    _, t_fwd, _ = wall(lambda: [model.engine.infer(win) for _ in range(6 * len(S))], 5)
    return {'datasets': len(S), 'orientations': 6, 'nfb': 32, 'precision': 'bf16', 'host_s': t_host, 'device_s': t_dev,
            'device_s_all': ts, 'forwards_114_s': t_fwd, 'speedup': t_host / t_dev, 'logs': dev,
            'pred_regions_min': int(min(nreg)), 'pred_regions_mean': float(np.mean(nreg)),
            'pred_regions_max': int(max(nreg)), 'equal_to_host': True}


def bench_fit(S, M, tmp):
    names = ['synthetic.%02d' % i for i in range(len(S))]
    out = {}
    for name in ('device', 'host', 'device_again'):
        np.random.seed(865)
        api = UNet2DSummary(cpdir=os.path.join(tmp, 'cp_' + name), dataset_name_func=lambda p: p,
                            series_summary_func=lambda p: S[names.index(p)], mask_summary_func=lambda p: M[names.index(p)],
                            net_builder_func=lambda shape: unet(shape, nb_filters_base=32, precision='bf16', seed=3))
        timing = {'validate_s': 0.}
        orig = api._validate

        def timed_validate(model, S_, M_, names, yc, sv, epoch, val=None):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if name == 'host':
                r = host_validate(model, S_, M_, yc, sv, epoch)[0]
            else:
                r = orig(model, S_, M_, names, yc, sv, epoch, val)
            timing['validate_s'] += time.perf_counter() - t0
            return r
        api._validate = timed_validate
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hist, _ = api.fit(names, shape_trn=(128, 128), shape_val=(512, 512), batch_size_trn=20, nb_steps_trn=100,
                          nb_epochs=1, prop_trn=0.75, prop_val=0.25)
        torch.cuda.synchronize()
        out[name] = {'fit_s': time.perf_counter() - t0, 'validate_s': timing['validate_s'],
                     'val_logs': {k: v[0] for k, v in hist.items() if k.startswith('val_')}}
    assert all(same(out['device']['val_logs'][k], out['host']['val_logs'][k]) for k in out['host']['val_logs'])
    out['note'] = ('summary images and masks are given as arrays (no dataset files, no _summarize_mask); fit_s includes '
                   'the first-call CUDA graph captures; device_again repeats the device run after the host run')
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'validation_b200.json'))
    ap.add_argument('--skip-fit', action='store_true')
    args = ap.parse_args()
    rng = np.random.default_rng(2024)
    res = {'gpu': gpu_info(), 'cpu_count': os.cpu_count()}
    res['scoring'] = bench_scoring(rng)
    print(json.dumps(res['scoring'], indent=1), flush=True)
    S, M = make_data(rng)
    res['validate'] = bench_validate(S, M)
    print(json.dumps(res['validate'], indent=1), flush=True)
    if not args.skip_fit:
        with tempfile.TemporaryDirectory() as tmp:
            res['fit_epoch'] = bench_fit(S, M, tmp)
        print(json.dumps(res['fit_epoch'], indent=1), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fp:
        json.dump(res, fp, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
