"""The reference arm of bench.py (`--impl reference`: the CPU oracle port timed on the host cores) runs without a GPU;
its JSON line must carry the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line(tmp_path):
    dump = tmp_path / 'outputs'
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
                          '--dump-outputs', str(dump)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['higher_is_better'] is True and d['unit'] == 'images/s'
    assert d['metric'] == 'UNet2DS 512x512 images/sec (8x TTA)' and d['steps'] == 1 and d['value'] > 0
    assert d['config']['workload'] and d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    # --dump-outputs: the last step's thresholded mask and averaged activation
    mask, act = np.load(dump / 'mask.npy'), np.load(dump / 'act.npy')
    assert mask.dtype == np.float32 and act.dtype == np.float64 and mask.shape == act.shape == (512, 512)
    assert np.array_equal(mask, (act > 0.5).astype(np.float32))


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '0'],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 2 and '--steps must be at least 1' in out.stderr
