"""Throughput of UNetEngine.predict_tiled (overlap-tile 8x TTA for summary images larger than the 512^2 window) against the
512^2 headline path (predict_tta), nfb 32, one GPU.

    python scripts/large_image_bench.py [--precision fp16] [--out profiles/large_image_fp16.json]

Per image size: images/s and device time per image (CUDA events around back-to-back graph replays, >= 1 s of work after
three warm-up calls: eager, capture, replay), computed / useful pixels of the tile plan, ns per useful pixel next to the
512^2 headline, and the peak of torch.cuda.max_memory_allocated while that size runs.  The activations of every size are
far larger than the 126 MB L2 except the 512^2 control, which is the headline configuration itself.  The GPU's name and
power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'deep-calcium_b200')); sys.path.insert(0, ROOT)
os.environ.setdefault('DEEP_CALCIUM_HOME', '/tmp/deep-calcium-home')
import numpy as np  # noqa: E402
import torch  # noqa: E402
from deepcalcium.engine.graph import GraphSpec, he_normal_weights, plan_tiles  # noqa: E402
from deepcalcium.engine.unet_engine import UNetEngine  # noqa: E402

SIZES = [(512, 512), (796, 512), (1024, 1024), (2048, 2048), (4096, 4096)]


def gpu_info():
    q = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()), '--query-gpu=name,power.limit',
                        '--format=csv,noheader'], capture_output=True, text=True)
    name, limit = (q.stdout.strip().split(', ') + [None, None])[:2] if q.returncode == 0 else (None, None)
    return {'torch_name': torch.cuda.get_device_name(), 'smi_name': name, 'power_limit': limit}


def timed(fn, min_seconds=1.0):
    """device ms per call of fn over back-to-back calls totalling at least min_seconds"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); e1.synchronize()
    reps = max(5, int(min_seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--precision', default='fp16')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'large_image_fp16.json'))
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    spec = GraphSpec(32)
    eng = UNetEngine(spec, precision=args.precision)
    eng.set_weights_dict(he_normal_weights(spec, seed=7535))
    rng = np.random.default_rng(0)
    res = {'gpu': gpu_info(), 'precision': args.precision, 'nfb': 32, 'augmentation': 8, 'halo': eng.halo,
           'tile_batch_pixels': eng.tile_batch_pixels, 'sizes': []}

    s512 = torch.from_numpy(rng.standard_normal((512, 512)).astype(np.float32)).cuda()
    torch.cuda.reset_peak_memory_stats()
    ms, reps = timed(lambda: eng.predict_tta(s512))
    headline_ns = ms * 1e6 / (512 * 512)
    res['headline_predict_tta_512'] = {'ms_per_image': ms, 'images_per_s': 1e3 / ms, 'ns_per_useful_pixel': headline_ns,
                                       'replays': reps, 'max_memory_allocated_GiB': torch.cuda.max_memory_allocated() / 2**30}
    print('headline predict_tta 512^2: %.3f ms/image' % ms, flush=True)
    for hs, ws in SIZES:
        s = torch.from_numpy(rng.standard_normal((hs, ws)).astype(np.float32)).cuda()
        plan = plan_tiles((hs, ws), eng.halo)
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        ms, reps = timed(lambda: eng.predict_tiled(s))
        row = {'shape': [hs, ws], 'tile': plan.tile, 'grid': list(plan.grid), 'canvas': list(plan.canvas),
               'computed_over_useful_pixels': plan.computed_pixels() / float(hs * ws),
               'ms_per_image': ms, 'images_per_s': 1e3 / ms, 'ns_per_useful_pixel': ms * 1e6 / (hs * ws),
               'ns_per_computed_pixel': ms * 1e6 / plan.computed_pixels(),
               'vs_headline_ns_per_pixel': ms * 1e6 / (hs * ws) / headline_ns, 'replays': reps,
               'max_memory_allocated_GiB': torch.cuda.max_memory_allocated() / 2**30}
        res['sizes'].append(row)
        print('%4d x %4d: tile %d grid %s, %.3f ms/image, %.3f ns/useful px (%.2fx headline), computed/useful %.3f, '
              'peak %.2f GiB' % (hs, ws, plan.tile, plan.grid, ms, row['ns_per_useful_pixel'], row['vs_headline_ns_per_pixel'],
                                 row['computed_over_useful_pixels'], row['max_memory_allocated_GiB']), flush=True)
    res['gpu_after'] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
