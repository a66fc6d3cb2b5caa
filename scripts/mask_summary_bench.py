"""What the truth-mask summary (_summarize_mask) costs on the host and on the device.

    python scripts/mask_summary_bench.py [--out profiles/mask_summary_b200.json] [--skip-evaluate]

(a) Device time of one dcb_mask_summary call (CUDA events over back-to-back calls, masks already on the device, workspace
    allocated once) on random disk neurons at 512^2 with n = 300, 800 and 3000, and on the worst case: two neurons
    interleaved as a checkerboard, where every pixel is a candidate of one cluster walked by one thread.  The masks
    (n * 256 KiB) exceed the 126 MB L2 from n = 800 on.
(b) _summarize_mask(dspath) wall time, ending in a device synchronise, on .hdf5 datasets of 300 and 800 neurons: the host
    function it replaced (oracle/masks.py: reads the whole dataset) against the default plugin, with the device path split
    into file read, upload of masks/raw, kernels and download.
(c) UNet2DSummary.evaluate (two predict passes, each scoring every dataset) over 19 synthetic 300-neuron 512^2 .hdf5
    datasets at nb_filters_base 32, fp16, with oracle.masks.summarize_mask as mask_summary_func against the default.
The device results must equal the host ones; the script checks that.  The GPU's name and power limit are read in the
same run.
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
sys.path.insert(0, os.path.join(ROOT, 'scripts')); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import mask_corpus as mc  # noqa: E402
from deepcalcium.datasets.nf import make_dataset, open_dataset, summarize_masks_device  # noqa: E402
from deepcalcium.engine import ops  # noqa: E402
from deepcalcium.models.neurons import UNet2DSummary, unet  # noqa: E402
from deepcalcium.models.neurons.unet_2d_summary import _summarize_mask  # noqa: E402
from large_image_bench import gpu_info, timed  # noqa: E402
from oracle.masks import summarize_mask, summarize_mask_array  # noqa: E402


def wall(fn, reps):
    torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        t.append(time.perf_counter() - t0)
    return out, float(np.median(t)), t


def bench_kernel(rng):
    out = {}
    cases = [('disks_%d' % n, mc.disks(rng, n, 512, 512)) for n in (300, 800, 3000)]
    cases.append(('checkerboard', mc.checkerboard(512, 512)))
    for name, m in cases:
        n, H, W = m.shape
        dev = torch.from_numpy(m).cuda()
        res = torch.empty(H, W, dtype=torch.uint8, device='cuda')
        ws = torch.empty(ops.mask_summary_workspace_bytes(n, H, W), dtype=torch.uint8, device='cuda')
        ops.mask_summary(dev, res, ws)
        assert np.array_equal(res.cpu().numpy().astype(np.float64), summarize_mask_array(m)), name
        _, ncand, sizes = mc.decomposed(m)
        ms, reps = timed(lambda: ops.mask_summary(dev, res, ws), 1.0)
        out[name] = {'n': n, 'shape': [H, W], 'candidates': ncand, 'clusters': len(sizes),
                     'largest_cluster': int(sizes.max()) if len(sizes) else 0, 'device_ms': ms, 'reps': reps,
                     'mask_bytes': int(m.nbytes), 'read_GBps': m.nbytes / (ms * 1e-3) / 1e9, 'bit_identical': True}
        print(name, json.dumps(out[name]), flush=True)
    return out


def bench_plugin(rng, tmp):
    out = {}
    for n in (300, 800):
        m = mc.disks(rng, n, 512, 512)
        mean = (rng.random((512, 512)) * 50 + m.max(0) * 100).astype(np.float32)
        p = make_dataset(os.path.join(tmp, 'plugin_%d.hdf5' % n), 'synthetic.%d' % n, mean=mean, mx=mean, masks=m)
        host, t_host, _ = wall(lambda: summarize_mask(p), 3)
        _summarize_mask(p)
        dev, t_dev, ts = wall(lambda: _summarize_mask(p), 5)
        assert dev.dtype == host.dtype and np.array_equal(dev, host)
        # the device path in its parts
        _, t_read, _ = wall(lambda: open_dataset(p, keys=('masks/raw',)), 5)
        raw = open_dataset(p, keys=('masks/raw',))['masks/raw']
        _, t_up, _ = wall(lambda: torch.from_numpy(raw).cuda(), 5)
        d = torch.from_numpy(raw).cuda()
        r, t_kern, _ = wall(lambda: summarize_masks_device(d), 5)
        _, t_down, _ = wall(lambda: r.cpu().numpy().astype(np.float64), 5)
        _, t_read_all, _ = wall(lambda: open_dataset(p), 3)
        out['neurons_%d' % n] = {'file_MB': os.path.getsize(p) / 1e6, 'host_s': t_host, 'device_s': t_dev,
                                 'device_s_all': ts, 'speedup': t_host / t_dev, 'read_masks_raw_s': t_read,
                                 'read_whole_dataset_s': t_read_all, 'upload_s': t_up,
                                 'upload_GBps': raw.nbytes / t_up / 1e9, 'kernels_incl_alloc_s': t_kern,
                                 'download_s': t_down, 'host_compute_s': t_host - t_read_all, 'equal_to_host': True}
        print(n, json.dumps(out['neurons_%d' % n]), flush=True)
    return out


def bench_evaluate(rng, tmp, count=19):
    paths = []
    for i in range(count):
        m = mc.disks(rng, 300, 512, 512)
        mean = (rng.standard_normal((512, 512)) * 20 + m.max(0) * 100).astype(np.float32)
        paths.append(make_dataset(os.path.join(tmp, 'eval_%02d.hdf5' % i), 'synthetic.%02d' % i, mean=mean, mx=mean,
                                  masks=m))
    model = unet((512, 512), nb_filters_base=32, precision='fp16', seed=3)
    out = {}
    for name, func in (('default', _summarize_mask), ('host', summarize_mask), ('default_again', _summarize_mask)):
        api = UNet2DSummary(cpdir=os.path.join(tmp, 'cp_' + name), mask_summary_func=func)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        scores = api.evaluate(paths, model)
        torch.cuda.synchronize()
        out[name] = {'evaluate_s': time.perf_counter() - t0, 'scores': {str(k): v for k, v in scores.items()}}
        print(name, json.dumps(out[name]), flush=True)
    assert json.dumps(out['default']['scores']) == json.dumps(out['host']['scores'])
    out['datasets'] = count
    out['note'] = ('two predict passes (8x TTA and none) with print_scores: mask_summary_func runs twice per dataset; '
                   'default_again repeats the default run after the host run')
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'mask_summary_b200.json'))
    ap.add_argument('--skip-evaluate', action='store_true')
    args = ap.parse_args()
    rng = np.random.default_rng(2026)
    res = {'gpu': gpu_info(), 'cpu_count': os.cpu_count()}
    res['kernel'] = bench_kernel(rng)
    with tempfile.TemporaryDirectory() as tmp:
        res['summarize_mask'] = bench_plugin(rng, tmp)
        if not args.skip_evaluate:
            res['evaluate'] = bench_evaluate(rng, tmp)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fp:
        json.dump(res, fp, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
