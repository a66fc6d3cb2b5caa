"""What nb_filters_base costs in the 16-bit modes, where widths other than 32 and 64 run on zero-padded channels
(engine/graph.py, padded_width).

    python scripts/width_bench.py [--out profiles/width_fp16_bf16.json]

For nb_filters_base in {8, 16, 24, 32, 48, 64} and both up-path modes:
  * fp16 8x TTA of one 512^2 summary image (predict_tta): device ms per image over back-to-back graph replays;
  * one bf16 training step on 32 crops of 128^2 (dice loss, Adam, dropout on; the C3 shape of bench.py): ms per step
    over graph replays;
  * GFLOP of both workloads on the real graph and on the padded graph that runs (GraphSpec.flops_forward / flops_train);
  * peak torch.cuda.max_memory_allocated of each workload.
The fp32 check mode at nb_filters_base 16 (the only way it ran before the padded layout) is timed on the same two
workloads for contrast.  Every timed window holds >= 1 s of work after three warm-up calls (eager, capture, replay).  The
GPU's name and power limit are read in the same run.
"""
import argparse
import gc
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'deep-calcium_b200')); sys.path.insert(0, ROOT)
os.environ.setdefault('DEEP_CALCIUM_HOME', '/tmp/deep-calcium-home')
sys.path.insert(0, os.path.join(ROOT, 'scripts'))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from deepcalcium.engine.graph import GraphSpec, he_normal_weights  # noqa: E402
from deepcalcium.engine.unet_engine import UNetEngine  # noqa: E402
from large_image_bench import gpu_info, timed  # noqa: E402

WIDTHS = [8, 16, 24, 32, 48, 64]
B, CROP, TTA = 32, 128, 8


def measure(nfb, mode, infer_precision, train_precision, rng):
    spec = GraphSpec(nfb, upsampling_or_transpose=mode)
    w = he_normal_weights(spec, seed=7535)
    row = {'nfb': nfb, 'mode': mode}
    s512 = torch.from_numpy(rng.standard_normal((512, 512)).astype(np.float32)).cuda()
    xs = [torch.from_numpy(rng.standard_normal((B, CROP, CROP)).astype(np.float32)).cuda() for _ in range(4)]
    ys = [torch.from_numpy((rng.random((B, CROP, CROP)) < 0.126).astype(np.uint8)).cuda() for _ in range(4)]
    for what, precision in (('tta512', infer_precision), ('train', train_precision)):
        gc.collect()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        eng = UNetEngine(spec, precision=precision)
        eng.set_weights_dict(w)
        if what == 'tta512':
            ms, reps = timed(lambda: eng.predict_tta(s512))
            flops = [TTA * sp.flops_forward(512, 512) for sp in (spec, eng.dspec)]
        else:
            k = [0]

            def step():
                k[0] += 1
                eng.train_step(xs[k[0] % 4], ys[k[0] % 4], loss='dice_loss', dropout=True)
            ms, reps = timed(step)
            flops = [B * sp.flops_train(CROP, CROP) for sp in (spec, eng.dspec)]
        row[what] = {'precision': precision, 'ms': ms, 'replays': reps, 'gflop_real': flops[0] / 1e9,
                     'gflop_padded': flops[1] / 1e9, 'tflops_real': flops[0] / ms / 1e9,
                     'max_memory_allocated_GiB': torch.cuda.max_memory_allocated() / 2 ** 30}
        del eng
    t, r = row['tta512'], row['train']
    print('nfb %2d %-10s | fp16 TTA 512^2 %7.3f ms (%.0f / %.0f GFLOP real / padded, %.1f GiB) | %s train 32x128^2 %7.3f ms '
          '(%.0f / %.0f GFLOP, %.1f GiB)' % (nfb, mode, t['ms'], t['gflop_real'], t['gflop_padded'], t['max_memory_allocated_GiB'],
                                            r['precision'], r['ms'], r['gflop_real'], r['gflop_padded'],
                                            r['max_memory_allocated_GiB']), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'width_fp16_bf16.json'))
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    rng = np.random.default_rng(0)
    res = {'gpu': gpu_info(), 'tta': TTA, 'train_batch': [B, CROP, CROP], 'loss': 'dice_loss', 'rows': []}
    for mode in ('transpose', 'upsampling'):
        for nfb in WIDTHS:
            res['rows'].append(measure(nfb, mode, 'fp16', 'bf16', rng))
    res['fp32_check_mode'] = measure(16, 'transpose', 'fp32', 'fp32', rng)
    res['gpu_after'] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
