#!/usr/bin/env python
"""Benchmark of the UNet2DS hot path (BASELINE.json metric: UNet2DS 512^2 images/sec with 8x TTA,
plus train crops/sec and the projection's GB/s as extra keys on the same JSON line).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels)
    python bench.py --impl reference --steps K --warmup W    # CPU arm: oracle port of the Keras graph

A step = one 512x512 summary image through the full 8x-TTA prediction on every rank (independent
images per rank: weak scaling, no data-path collective).  `value` is device-timed with the input
already in HBM; `e2e` goes through UNet2DSummary.predict with host buffers in and the mask out.

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/mask.npy (float32 0/1) and
DIR/act.npy (float64, the 8x-TTA averaged probability); inputs and weights are seeded, so two builds run
with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, 'deep-calcium_b200'), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)
os.environ.setdefault('DEEP_CALCIUM_HOME', '/tmp/deep-calcium-home')
# torchrun exports OMP_NUM_THREADS=1; the CPU legs (rank 0 only) are entitled to every core this process may use, and the
# OpenMP pool is sized when torch is first imported - so this has to happen before that import
try:
    _HOST_CORES = max(1, len(os.sched_getaffinity(0)))
except Exception:   # noqa: BLE001
    _HOST_CORES = os.cpu_count() or 1
if int(os.environ.get('RANK', '0')) == 0:
    os.environ['OMP_NUM_THREADS'] = str(_HOST_CORES)
    os.environ['MKL_NUM_THREADS'] = str(_HOST_CORES)

import numpy as np  # noqa: E402

METRIC = 'UNet2DS 512x512 images/sec (8x TTA)'
WORKLOAD = 'unet2ds_512x512_tta8_nfb32_random_init'


def peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            p = json.load(f)
        return dict(hbm=float(p['hbm_gbs']), tf=float(p['bf16_tflops']), tf_sus=float(p['bf16_tflops_sustained']),
                    src='measured (MEASURED_PEAKS.json)')
    except Exception:
        return dict(hbm=6650.0, tf=1590.0, tf_sus=1400.0, src='fallback (B200_PROFILING.md)')


class ClockSampler(object):
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(',')]))

    def samples_inside(self, t0, t1):
        return sum(1 for t, r in list(self.rows) if len(r) >= 7 and r[0].replace('.', '').isdigit() and t0 - 0.02 <= t <= t1 + 0.02)

    def stop(self, window=None):
        """window = (t0, t1) wall-clock bounds of the timed region.  The sampler runs from before the warm-up until
        after the end-to-end arm (the GPU is under the same load throughout); samples inside the timed region are
        preferred, and when that region is shorter than nvidia-smi's sampling period all samples under load are used."""
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [(t, r) for t, r in self.rows if len(r) >= 7 and r[0].replace('.', '').isdigit()]
        scope = 'whole run under load (warm-up, timed region, e2e arm)'
        if window is not None:
            inside = [(t, r) for t, r in rows if window[0] - 0.02 <= t <= window[1] + 0.02]
            if len(inside) >= 3:
                rows, scope = inside, 'timed region'
        sm = [float(r[0]) for _, r in rows]
        mx = [float(r[1]) for _, r in rows if r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for _, r in rows for i in range(4) if r[3 + i].lower() == 'active'})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm), 'sampled_over': scope}


# ---------------------------------------------------------------------------------------------- CPU arm
def cpu_forward_tta(w, s, spec, n_images):
    """oracle port of predict(augmentation=True) (unet_2d_summary.py:585-595) in float32 on all host cores
    -> (seconds, (mask, act) of the last image)"""
    import torch
    import oracle
    torch.set_num_threads(_HOST_CORES)
    t0 = time.perf_counter()
    for _ in range(n_images):
        out = oracle.tta_predict(w, s, spec, augmentation=True, dtype=torch.float32)
    return time.perf_counter() - t0, out


def dump_outputs(path, mask, act):
    """--dump-outputs: the arrays the timed path returned in its last step"""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, 'mask.npy'), np.asarray(mask, dtype=np.float32))
    np.save(os.path.join(path, 'act.npy'), np.asarray(act, dtype=np.float64))


def run_reference(args):
    import torch
    import oracle
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    spec = oracle.UNetSpec(32)
    w = oracle.init_weights(spec, seed=7535)
    s = np.random.default_rng(865).standard_normal((512, 512)).astype(np.float32)
    for _ in range(min(args.warmup, 1)):
        cpu_forward_tta(w, s, spec, 1)
    dt, (mask, act) = cpu_forward_tta(w, s, spec, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, mask, act)
    val = args.steps / dt
    cores = torch.get_num_threads()
    line = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'images/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': min(args.warmup, 1), 'ms_per_step': 1e3 * dt / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'window': 512, 'tta': 8, 'weights': 'random-init seed 7535'},
            'cpu_baseline': {'value': val, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                             'sample': '%d TTA images (8 forwards each) of the torch-CPU fp32 oracle port of the Keras '
                                       'graph; Keras 2.0.6/TF 1.2.1 are not installable' % args.steps},
            'e2e': {'value': val, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))



# ---------------------------------------------------------------------------------------------- parity (outside the timed regions)
def parity_inference(eng, w, img_dev, precision):
    """The benchmarked image under the exact dispatch that was timed (same engine, same captured graph) against the
    CPU oracle: 8x-TTA mask disagreement (north star: <= 0.1 %) and logit error of the identity-transform forward
    (north star: 1e-2 abs in 16-bit mode, 1e-4 in the fp32 check mode)."""
    import torch
    import oracle
    ospec = oracle.UNetSpec(32)
    s = img_dev.cpu().numpy()
    mask, _ = eng.predict_tta(img_dev)
    mask = mask.cpu().numpy().copy()
    logit = eng._session(8, 512, 512, False)['logit'][0].cpu().numpy().copy()      # transform 0 = identity
    omask, _ = oracle.tta_predict(w, s, ospec, dtype=torch.float32)
    with torch.no_grad():
        ologit = oracle.unet_forward(w, s[None], ospec, dtype=torch.float64)['logit'][0].numpy()
    err = np.abs(logit - ologit)
    tol = 1e-4 if precision == 'fp32' else 1e-2
    return {'oracle': 'CPU restatement of the Keras graph (oracle/, parity unpinned)', 'image': 'benchmark image 0',
            'mask_disagreement': float(np.mean(mask != omask)), 'mask_tolerance': 1e-3,
            'logit_max_abs_err': float(err.max()), 'logit_mean_abs_err': float(err.mean()), 'logit_tolerance': tol,
            'logit_range': float(np.abs(ologit).max()),
            'pass': bool(np.mean(mask != omask) <= 1e-3 and err.max() <= tol)}


def parity_train(precision, w, x_dev, y_dev):
    """One train_on_batch of the benchmarked batch (dropout off) on a fresh engine under the default dispatch: loss and
    every gradient tensor against oracle.train_step (float64); in bf16 mode also the oracle's own bf16-storage emulation
    as the yardstick of what 8-bit mantissas can give on this network."""
    import oracle
    from deepcalcium.engine.graph import GraphSpec
    from deepcalcium.engine.unet_engine import UNetEngine
    ospec = oracle.UNetSpec(32)
    x, y = x_dev.cpu().numpy(), y_dev.cpu().numpy()
    L, _, _, g, _ = oracle.train_step(w, x, y, spec=ospec, loss='dice_loss')
    eng = UNetEngine(GraphSpec(32), precision=precision)
    eng.set_weights_dict(w)
    m = eng.train_step(x_dev, y_dev, loss='dice_loss', lr=0.002, dropout=False)

    def rel(a, b):
        return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))

    keys = [k for k in g if not (k.endswith('/bias') and not k.startswith('head'))]
    errs = {k: rel(eng.G[k].cpu().numpy().astype(np.float64), g[k]) for k in keys}
    worst = max(errs, key=errs.get)
    out = {'loss': float(m[0].item()), 'oracle_loss': L, 'loss_abs_err': abs(float(m[0].item()) - L),
           'grad_rel_l2_err_worst': errs[worst], 'grad_rel_l2_err_worst_tensor': worst,
           'grad_rel_l2_err_median': float(np.median(list(errs.values()))), 'dropout': 'off for the parity step'}
    if precision != 'fp32':
        g_emu = oracle.train_step(w, x, y, spec=ospec, loss='dice_loss', emulate_bf16=True)[3]
        emu = {k: rel(g_emu[k], g[k]) for k in keys}
        out['bf16_storage_emulation_grad_rel_l2_err_worst'] = max(emu.values())
        out['bf16_storage_emulation_grad_rel_l2_err_median'] = float(np.median(list(emu.values())))
        out['pass'] = bool(out['loss_abs_err'] < 2e-3 and all(errs[k] <= 1.3 * emu[k] + 0.03 for k in keys))
    else:
        out['pass'] = bool(out['loss_abs_err'] < 1e-4 and errs[worst] < 3e-3)
    return out


# ---------------------------------------------------------------------------------------------- CPU baselines (rank 0, N = 1)
def cpu_baselines(w, img_host):
    """The CPU legs BASELINE.md section 3 lists, each on a bounded sample, all host cores unless stated."""
    import torch
    import oracle
    ospec = oracle.UNetSpec(32)
    out = {}
    cores = torch.get_num_threads()
    # 8x TTA inference (the headline metric)
    cpu_forward_tta(w, img_host[:128, :128].copy(), ospec, 1)
    n_cpu = 2
    dt = cpu_forward_tta(w, img_host, ospec, n_cpu)[0]
    head = {'value': n_cpu / dt, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
            'sample': '%d TTA images (16 fp32 forwards) of the torch-CPU oracle port of the Keras graph' % n_cpu}
    # training step (fwd + bwd + Keras-Adam), fp32, the C3 batch
    rng = np.random.default_rng(865)
    x = rng.standard_normal((32, 128, 128)).astype(np.float32)
    y = (rng.random((32, 128, 128)) < 0.126).astype(np.uint8)
    t0 = time.perf_counter()
    oracle.train_step(w, x, y, spec=ospec, loss='dice_loss', dtype=torch.float32)
    dt = time.perf_counter() - t0
    out['train_step'] = {'value': 32 / dt, 'unit': 'crops/s', 'cores': cores, 'kind': 'port',
                         'sample': '1 step of 32 crops 128x128 (fwd + autograd + Keras-Adam, torch-CPU fp32)'}
    # projection: (i) numpy mean(float64)+max, 1 thread; (ii) the faithful per-frame loop of nf.py:126-130 (float16
    # read-modify-write mean, int16 running max) on an in-memory array; (iii) a multi-threaded torch reduction
    T = 300
    sub = (np.random.default_rng(7535).random((T, 512, 512), dtype=np.float32) * 4096).astype(np.float32)
    t0 = time.perf_counter(); sub.mean(0, dtype=np.float64); sub.max(0); dt = time.perf_counter() - t0
    out['projection_numpy'] = {'value': sub.nbytes / dt / 1e9, 'unit': 'GB/s', 'cores': 1, 'kind': 'port',
                               'sample': '%d of 3000 frames, numpy mean(float64) + max' % T}
    sub16 = sub[:100].astype(np.int16)
    t0 = time.perf_counter(); oracle.project_streaming_fp16(sub16); dt = time.perf_counter() - t0
    out['projection_reference_loop'] = {'value': 100 / dt, 'unit': 'frames/s', 'cores': 1, 'kind': 'port',
                                        'sample': '100 int16 frames through the per-frame loop of datasets/nf.py:126-130 '
                                                  '(in-memory arrays; the reference reports ~205 frames/s with TIFF + HDF5 I/O)'}
    tt = torch.from_numpy(sub)
    t0 = time.perf_counter(); tt.to(torch.float64).mean(0); tt.amax(0); dt = time.perf_counter() - t0
    out['projection_torch_mt'] = {'value': sub.nbytes / dt / 1e9, 'unit': 'GB/s', 'cores': cores, 'kind': 'port',
                                  'sample': '%d of 3000 frames, torch float64 mean + amax' % T}
    return head, out


# ---------------------------------------------------------------------------------------------- GPU arm
def ncu_conv_traffic(precision):
    """DRAM traffic of the conv launches of ONE 8-image forward, measured in this run: `ncu --metrics dram__bytes_*` around
    scripts/profile_step.py (same engine, same weights, eager launches) as a subprocess, outside every timed region.
    Returns (bytes per step, per-kernel rows, description) or None when ncu is unavailable / fails (DCB_BENCH_NCU=0 skips it)."""
    import csv
    import io
    import shutil
    import subprocess
    if os.environ.get('DCB_BENCH_NCU', '1') == '0' or shutil.which('ncu') is None:
        return None
    metrics = 'dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active'
    cmd = ['ncu', '--metrics', metrics, '--clock-control', 'none', '--csv', '-k', 'regex:tapgemm_tc|conv3x3_c1_fwd',
           sys.executable, os.path.join(ROOT, 'scripts', 'profile_step.py'), 'infer', {'fp16': 'f16'}.get(precision, precision)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get(
            'CUDA_VISIBLE_DEVICES', '0'))).stdout
    except Exception:   # noqa: BLE001
        return None
    lines = [ln for ln in out.splitlines() if ln.startswith('"')]
    if len(lines) < 2:
        return None
    rows = list(csv.DictReader(io.StringIO('\n'.join(lines))))
    per = {}
    order = []
    for r in rows:
        kid = r['ID']
        if kid not in per:
            per[kid] = {'kernel': r['Kernel Name'].split('(')[0].replace('void dcb::', '').replace('dcb::', '')[:40]}
            order.append(kid)
        v = float(r['Metric Value'].replace(',', ''))
        u = r['Metric Unit']
        scale = {'Gbyte': 1e9, 'Mbyte': 1e6, 'Kbyte': 1e3, 'byte': 1.0, 'us': 1.0, 'ns': 1e-3, 'ms': 1e3, 'msecond': 1e3, 'usecond': 1.0,
                 'nsecond': 1e-3, 'second': 1e6}.get(u, 1.0)
        per[kid][r['Metric Name']] = v * scale
    if len(order) % 3 != 0:          # profile_step.py runs three identical steps
        return None
    last = order[-(len(order) // 3):]
    klist, tot = [], 0.0
    for kid in last:
        d = per[kid]
        rd, wr = d.get('dram__bytes_read.sum', 0.0), d.get('dram__bytes_write.sum', 0.0)
        tot += rd + wr
        klist.append({'kernel': d['kernel'], 'us': round(d.get('gpu__time_duration.sum', 0.0), 1), 'dram_read_MB': round(rd / 1e6, 1),
                      'dram_write_MB': round(wr / 1e6, 1),
                      'tensor_pipe_active_pct': round(d.get('sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active', 0.0), 1)})
    return tot, klist, ('measured in this run: ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum around the %d conv launches of one '
                        'eager 8-image forward (scripts/profile_step.py, subprocess, outside the timed regions)' % len(last))


def per_layer_profile(eng, sess, spec, NB, H, W, in_graph=False):
    """device time of every contraction launch of one forward pass, average of 5 passes -> (rows, total conv flops,
    total conv ms).  CUDA events on the launch stream around every launch: eager launches (each interval then includes the
    front-end latency of an individually submitted kernel), or - in_graph - EXTERNAL event-record nodes captured between the
    kernels of one CUDA graph of the forward pass, i.e. the launches as the timed region runs them (graph-launched), minus
    the programmatic overlap of neighbouring kernels, which an event node between them rules out."""
    import torch
    from deepcalcium.engine import ops
    rows = []
    orig = {}
    names = ['conv3x3_fwd', 'conv3x3_fwd_fused', 'convT2x2_fwd', 'conv3x3_c1_fwd', 'maxpool2x2', 'head_fwd']
    events = []

    def wrap(name):
        f = getattr(ops, name)
        orig[name] = f

        def g(*a, **k):
            e0 = torch.cuda.Event(enable_timing=True, external=in_graph)
            e1 = torch.cuda.Event(enable_timing=True, external=in_graph)
            e0.record()
            f(*a, **k)
            e1.record()
            events.append((name, a, e0, e1))
        setattr(ops, name, g)

    for n in names:
        wrap(n)
    passes = []                      # 2 warm-up passes, then the per-launch AVERAGE over 5 passes
    try:
        if in_graph:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                eng._forward_inference(sess)
            for it in range(7):
                g.replay()
                torch.cuda.synchronize()
                if it >= 2:
                    passes.append([e0.elapsed_time(e1) for _, _, e0, e1 in events])
        else:
            for it in range(7):
                del events[:]
                eng._forward_inference(sess)
                torch.cuda.synchronize()
                if it >= 2:
                    passes.append([e0.elapsed_time(e1) for _, _, e0, e1 in events])
    finally:
        for n, f in orig.items():
            setattr(ops, n, f)
    tot_f, tot_ms = 0.0, 0.0
    for li, (name, a, e0, e1) in enumerate(events):
        ms = float(np.mean([p[li] for p in passes]))
        fl = 0.0
        if name in ('conv3x3_fwd', 'conv3x3_fwd_fused'):
            src0, src1, wgt, out = a[0], a[1], a[2], a[3]
            cin = src0.shape[3] + (src1.shape[3] if src1 is not None else 0)
            fl = 2.0 * out.shape[0] * out.shape[1] * out.shape[2] * 9 * cin * out.shape[3]
            tag = 'conv3x3%s %dx%d %d->%d' % ('+fused' if name.endswith('fused') else '', out.shape[1], out.shape[2], cin, out.shape[3])
        elif name == 'convT2x2_fwd':
            src, out = a[0], a[2]
            fl = 2.0 * src.shape[0] * src.shape[1] * src.shape[2] * 4 * src.shape[3] * out.shape[3]
            tag = 'convT2x2 %dx%d %d->%d' % (src.shape[1], src.shape[2], src.shape[3], out.shape[3])
        else:
            tag = name
        if fl:
            tot_f += fl
            tot_ms += ms
        rows.append({'op': tag, 'ms': round(ms, 4), 'tflops': round(fl / ms / 1e9, 1) if fl else None})
    return rows, tot_f, tot_ms


def run_ours(args):
    import torch
    import torch.distributed as dist
    from deepcalcium import _native as nat
    from deepcalcium.engine.graph import GraphSpec
    from deepcalcium.engine.unet_engine import UNetEngine
    from deepcalcium.engine.graph import he_normal_weights

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    dev = torch.device('cuda', local)
    pk = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    spec = GraphSpec(32)
    w = he_normal_weights(spec, seed=7535)
    rng = np.random.default_rng(7535)
    for blk in spec.blocks:          # randomised BN statistics so that the folded BN is not the identity
        if blk.kind != 'head':
            w[blk.name + '/moving_mean'] = (0.1 * rng.standard_normal(blk.cout)).astype(np.float32)
            w[blk.name + '/moving_var'] = rng.uniform(0.5, 1.5, blk.cout).astype(np.float32)
    eng = UNetEngine(spec, precision=args.precision)
    eng.set_weights_dict(w)
    n_img = 4
    imgs = [torch.from_numpy(np.random.default_rng(865 + rank * 100 + i).standard_normal((512, 512)).astype(np.float32)).to(dev)
            for i in range(n_img)]

    # ---- kernel-only arm: inputs resident in HBM, device-timed
    sampler = ClockSampler(local)
    sampler.start()
    for i in range(max(args.warmup, 3)):
        eng.predict_tta(imgs[i % n_img])
    # keep the GPU under the same load until nvidia-smi has started reporting (its first sample takes ~100 ms)
    t_load = time.time()
    while not sampler.rows and time.time() - t_load < 1.0:
        eng.predict_tta(imgs[0])
        torch.cuda.synchronize()
    barrier()
    launches0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_w0 = time.time()
    e0.record()
    for i in range(args.steps):
        mask, act = eng.predict_tta(imgs[i % n_img])
    e1.record()
    barrier()
    t_w1 = time.time()
    # predict_tta returns static buffers, which the end-to-end arm below overwrites
    last = (mask.cpu().numpy(), act.cpu().numpy()) if args.dump_outputs and rank == 0 else None
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = eng.launches - launches0
    value = world * args.steps / (ms / 1e3)
    # nvidia-smi polling takes the driver lock for a fraction of a millisecond per query and shows up in the host-synchronous
    # end-to-end arm (1069 vs 1096 images/s): once the timed region holds enough samples the sampler is stopped here
    clocks = None
    time.sleep(0.03)                 # let the reader thread take in the last samples of the timed region
    if sampler.samples_inside(t_w0, t_w1) >= 3:
        clocks = sampler.stop(window=(t_w0, t_w1))

    # ---- e2e arm: the reference-facing API with host buffers (UNet2DSummary.predict, :532)
    from deepcalcium.models.neurons import UNet2DSummary
    from deepcalcium.models.neurons.unet_2d_summary import UNetModel
    host_imgs = {('img%d' % i): imgs[i].cpu().numpy() for i in range(n_img)}
    model = UNetModel.__new__(UNetModel)
    model.window_shape, model.spec, model.engine = (512, 512), spec, eng
    api = UNet2DSummary(cpdir='/tmp/deep-calcium-bench-cp-%d' % rank, dataset_name_func=lambda p: p,
                        series_summary_func=lambda p: host_imgs[p])
    paths = [('img%d' % (i % n_img)) for i in range(args.steps)]
    api.predict(paths[:6], model, augmentation=True)      # both pipeline slots warm (eager pass + graph capture each)
    barrier()
    t0 = time.perf_counter()
    Mp, _ = api.predict(paths, model, augmentation=True)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    if clocks is None:               # short timed region: all samples under load, end-to-end arm included
        clocks = sampler.stop(window=(t_w0, t_w1))
    e2e = {'value': world * args.steps / e2e_s, 'unit': 'images/s', 'h2d_bytes_per_step': 512 * 512 * 4,
           'd2h_bytes_per_step': int(Mp[0].nbytes)}

    line = {'metric': METRIC, 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': {'fp16': 'f16', 'bf16': 'bf16', 'fp32': 'f32'}[args.precision], 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'window': 512, 'tta': 8, 'batch_per_step': 8,
                       'weights': 'random-init he_normal seed 7535', 'parallelism': 'independent images per rank',
                       'l2': 'per-step activation footprint ~1.2 GB >> 126 MB L2; 4 rotating inputs'},
            'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches)}

    # ---- multi-GPU extras (every rank takes part in the collectives)
    dist_extra = {}
    if world > 1:
        for name, fn in (('tta_sharded', bench_tta_sharded), ('train_dp', bench_train_dp),
                         ('projection_sharded', bench_projection_sharded)):
            try:
                dist_extra[name] = fn(args, pk, eng, imgs, max_over_ranks, barrier)
            except Exception as ex:   # noqa: BLE001
                dist_extra[name] = {'error': repr(ex)}
    if rank == 0:
        # ---- roofline of the dominant kernel family (the conv tap-GEMMs), timed live with CUDA events
        try:
            sess = eng._session(8, 512, 512, False)
            rows_eager, tot_f, tot_ms_eager = per_layer_profile(eng, sess, spec, 8, 512, 512)
            how = 'event-record nodes between the kernels of one captured forward pass (graph-launched, like the timed region)'
            try:
                rows, tot_f, tot_ms = per_layer_profile(eng, sess, spec, 8, 512, 512, in_graph=True)
                if not (0.3 * tot_ms_eager < tot_ms < 1.5 * tot_ms_eager):
                    raise RuntimeError('implausible in-graph event timing: %.4f ms vs %.4f ms eager' % (tot_ms, tot_ms_eager))
                for r, re_ in zip(rows, rows_eager):
                    r['ms_eager'] = re_['ms']
            except Exception as ex:   # noqa: BLE001
                sys.stderr.write('per-layer timing inside a graph failed (%r); eager per-launch events instead\n' % (ex,))
                rows, tot_ms, how = rows_eager, tot_ms_eager, 'eager launches (front-end launch latency of every kernel included)'
            ach = tot_f / tot_ms / 1e9
            traffic, traffic_src, traffic_kernels = None, None, None
            live = ncu_conv_traffic(args.precision) if world == 1 else None
            if live is not None:
                traffic, traffic_kernels, traffic_src = live
            for name in (() if live is not None else ('r2_conv_traffic.json', 'r1_conv_traffic.json')):
                try:   # dram__bytes_read.sum + dram__bytes_write.sum over the same tensor-core launches (ncu --set full capture)
                    with open(os.path.join(ROOT, 'profiles', name)) as f:
                        traffic = json.load(f)['dram_bytes_per_step']
                    traffic_src = 'profiles/' + name + ' (ncu capture of this command; not re-measured in the run)'
                    break
                except Exception:   # noqa: BLE001
                    pass
            step_tf = 8 * spec.flops_forward(512, 512) / (ms / args.steps) / 1e9
            line['roofline'] = {'bound': 'tensor', 'achieved': ach, 'peak': pk['tf'], 'unit': 'TFLOP/s',
                                'frac': ach / pk['tf'], 'traffic': traffic, 'traffic_source': traffic_src,
                                'peak_source': pk['src'] + ', burst figure',
                                'kernel': 'tcgen05 tap-GEMM conv3x3/convT2x2 launches of one 8-image forward, each timed with '
                                          'CUDA events (per_layer, average of 5 passes): ' + how,
                                'flops_per_step': tot_f, 'conv_ms_per_step': tot_ms,
                                'conv_ms_per_step_eager_launches': tot_ms_eager, 'frac_eager_launches': tot_f / tot_ms_eager / 1e9 / pk['tf'],
                                'whole_step_tflops': step_tf, 'whole_step_frac_of_burst_peak': step_tf / pk['tf'],
                                'whole_step_frac_of_sustained_peak': step_tf / pk['tf_sus'],
                                'note': 'conv_ms_per_step sums the conv launches only; ms_per_step is the CUDA-graph replay of the '
                                        'whole step (all kernels incl. first layer, TTA batch/combine, programmatic overlap of '
                                        'neighbouring kernels)'}
            line['per_layer'] = rows
            if traffic_kernels is not None:
                line['roofline']['ncu_launches'] = traffic_kernels
        except Exception as ex:   # noqa: BLE001
            line['roofline'] = {'error': repr(ex)}
        # ---- parity of exactly what was timed (outside the timed region)
        try:
            line['parity'] = {'inference': parity_inference(eng, w, imgs[0], args.precision)}
        except Exception as ex:   # noqa: BLE001
            line['parity'] = {'inference': {'error': repr(ex)}}
        # ---- extras: projection (C2) and training (C3)
        line['extra'] = dict(dist_extra)
        if args.precision == 'fp16' and world == 1:
            try:      # the same step with bf16 storage (same MMA rate; its logit error is the reason fp16 is the default)
                line['extra']['inference_bf16'] = bench_inference_other(args, spec, w, imgs, 'bf16')
            except Exception as ex:   # noqa: BLE001
                line['extra']['inference_bf16'] = {'error': repr(ex)}
        for name, fn in (('projection', bench_projection), ('train', bench_train)):
            try:
                line['extra'][name] = fn(args, pk)
            except Exception as ex:   # noqa: BLE001
                line['extra'][name] = {'error': repr(ex)}
        if isinstance(line['extra'].get('train'), dict) and 'parity' in line['extra']['train']:
            line['parity']['train'] = line['extra']['train'].pop('parity')
        # ---- CPU baselines on this box's host cores (bounded samples; N = 1 only: at N > 1 the other ranks would idle)
        if world == 1:
            try:
                line['cpu_baseline'], line['extra']['cpu_baselines'] = cpu_baselines(w, imgs[0].cpu().numpy())
            except Exception as ex:   # noqa: BLE001
                line['cpu_baseline'] = {'error': repr(ex)}
        else:
            line['cpu_baseline'] = None
        if last is not None:
            dump_outputs(args.dump_outputs, *last)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bench_inference_other(args, spec, w, imgs, precision):
    import torch
    from deepcalcium.engine.unet_engine import UNetEngine
    eng = UNetEngine(spec, precision=precision)
    eng.set_weights_dict(w)
    for i in range(4):
        eng.predict_tta(imgs[i % len(imgs)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        eng.predict_tta(imgs[i % len(imgs)])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    par = parity_inference(eng, w, imgs[0], precision)
    return {'images_per_s': 1e3 / ms, 'ms_per_step': ms, 'parity': par}


def bench_tta_sharded(args, pk, eng, imgs, max_over_ranks, barrier):
    """BASELINE config C4: ONE 512x512 image, its 8 TTA transforms sharded over the ranks, probability maps
    gathered to rank 0 (NCCL all_gather over NVLink), fixed-order combine -> latency per image."""
    import torch
    from deepcalcium.engine.dist import Comm, predict_tta_sharded
    comm = Comm()
    for i in range(4):
        predict_tta_sharded(eng, imgs[0], comm)
    barrier()
    n = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        predict_tta_sharded(eng, imgs[i % len(imgs)], comm)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / n
    # parity: the sharded mask / activation against the single-GPU 8x TTA of the same image on rank 0
    mask, act = predict_tta_sharded(eng, imgs[1], comm)
    same = None
    if comm.rank == 0:
        mask, act = mask.clone(), act.clone()
        m1, a1 = eng.predict_tta(imgs[1])
        same = bool(torch.equal(mask, m1)) and bool(torch.equal(act, a1))
    barrier()
    return {'ms_per_image': ms, 'images_per_s': 1e3 / ms, 'ranks': comm.world, 'bit_identical': same,
            'nvlink_bytes_algorithmic': (8 - 8 // comm.world) * 512 * 512 * 4,
            'note': 'strong scaling of one image: transforms k -> rank k*n/8, probability maps to rank 0, fixed-order combine'}


def bench_train_dp(args, pk, eng_unused, imgs, max_over_ranks, barrier):
    """BASELINE config C5: data-parallel training, 32 crops of 128x128 per GPU, SyncBN + loss sums + gradient
    all-reduce (31 MB fp32) over NCCL."""
    import torch
    from deepcalcium.engine.graph import GraphSpec, he_normal_weights
    from deepcalcium.engine.unet_engine import UNetEngine
    from deepcalcium.engine.dist import Comm, sync_parameters, attach_peers
    comm = Comm()
    spec = GraphSpec(32)
    # the NCCL all-reduces (torch.distributed) are captured into the step's CUDA graph together with the kernels;
    # DCB_DP_GRAPHS=0 falls back to eager launches
    graphs = os.environ.get('DCB_DP_GRAPHS', '1') == '1'
    rng = np.random.default_rng(865 + comm.rank)
    B = 32
    x = torch.from_numpy(rng.standard_normal((B, 128, 128)).astype(np.float32)).cuda()
    y = torch.from_numpy((rng.random((B, 128, 128)) < 0.126).astype(np.uint8)).cuda()

    def make(use_graphs):
        eng = UNetEngine(spec, precision=train_precision(args), use_graphs=use_graphs)
        eng.set_weights_dict(he_normal_weights(spec, seed=7535))
        eng.comm = comm
        if os.environ.get('DCB_DP_PEERS', '1') == '1':
            attach_peers(eng, comm)          # SyncBN / loss sums exchanged inside the kernels over NVLink (no per-layer NCCL call)
        sync_parameters(eng, comm)
        for i in range(4):
            eng.train_step(x, y, loss='dice_loss', lr=0.002, dropout=True)
        torch.cuda.synchronize()
        return eng
    try:
        eng = make(graphs)
    except Exception as ex:   # noqa: BLE001 - capture of the collectives not supported by this torch/NCCL build
        sys.stderr.write('train_dp: graph capture failed (%r), eager launches instead\n' % (ex,))
        graphs = False
        eng = make(False)
    barrier()
    n = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        eng.train_step(x, y, loss='dice_loss', lr=0.002, dropout=True)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / n
    res = {'crops_per_s': comm.world * B * 1e3 / ms, 'ms_per_step': ms, 'global_batch': comm.world * B, 'ranks': comm.world,
           'launch': 'one CUDA graph per step, collectives captured' if graphs else 'eager (collectives interleaved)',
           'sync_bn': 'in-kernel peer exchange over NVLink (44 per step) + loss sums' if eng.peers is not None else 'NCCL all-reduce per layer',
           'grad_allreduce': 'one NCCL all-reduce of the flat 31 MB fp32 buffer after the backward pass (inside the step graph)'}
    del eng
    try:
        res.update(parity_train_dp(comm, spec))
    except Exception as ex:   # noqa: BLE001
        res['parity_error'] = repr(ex)
    return res


def parity_train_dp(comm, spec):
    """fp32 check mode, dropout off: one data-parallel step over a global batch of 4 x world crops of 64x64 against the
    single-device step on the concatenated batch (rank 0): loss and all-reduced gradients."""
    import torch
    from deepcalcium.engine.graph import he_normal_weights
    from deepcalcium.engine.unet_engine import UNetEngine
    from deepcalcium.engine.dist import shard_range, sync_parameters, attach_peers
    w = he_normal_weights(spec, seed=7535)
    Bg, H = 4 * comm.world, 64
    x = np.random.default_rng(1).standard_normal((Bg, H, H)).astype(np.float32)
    y = (np.random.default_rng(2).random((Bg, H, H)) < 0.126).astype(np.uint8)
    f, c = shard_range(Bg, comm.world, comm.rank)
    dp = UNetEngine(spec, precision='fp32', use_graphs=False)
    dp.set_weights_dict(w)
    dp.comm = comm
    if os.environ.get('DCB_DP_PEERS', '1') == '1':
        attach_peers(dp, comm)
    sync_parameters(dp, comm)
    m = dp.train_step(torch.from_numpy(x[f:f + c]).cuda(), torch.from_numpy(y[f:f + c]).cuda(), loss='dice_loss', dropout=False)
    loss_dp = float(m[0].item())
    out = {}
    if comm.rank == 0:
        from deepcalcium import _native as nat

        def single(**pol):
            ref = UNetEngine(spec, precision='fp32', use_graphs=False)
            ref.set_weights_dict(w)
            with nat.policy(**pol):
                loss = float(ref.train_step(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), loss='dice_loss', dropout=False)[0].item())
            worst = ('', 0.0)
            for k in dp.G:
                a_, b_ = dp.G[k].double().cpu().numpy(), ref.G[k].double().cpu().numpy()
                nb = np.linalg.norm(b_)
                r = float(np.linalg.norm(a_ - b_) / nb) if nb > 0 else float(np.abs(a_).max())
                if r > worst[1]:
                    worst = (k, r)
            wd, wr = dp.get_weights_dict(), ref.get_weights_dict()
            return loss, worst, max(float(np.max(np.abs(wd[k] - wr[k]))) for k in wd if 'moving' in k)
        # The data-parallel BatchNorm runs on the grid-barrier kernels with the in-kernel rank exchange, a single device picks the
        # channel-slab cluster kernels for its small tensors.  In the fp32 check mode every BatchNorm sum is an EXACT fixed-point
        # integer sum (csrc/bn_fused.cu: to_q40 / to_q20), so neither the kernel family nor the split of the batch over ranks
        # changes a single bit of it: grad_rel_err is measured against the single device on its DEFAULT dispatch; the figure
        # against the grid-barrier kernels on the single device (bn_slab = 0) is reported beside it.
        loss_ref, worst, stat = single()
        _, worst_g, _ = single(bn_slab=0)
        out = {'loss_abs_err': abs(loss_dp - loss_ref), 'grad_rel_err': worst[1], 'grad_rel_err_tensor': worst[0],
               'bn_moving_stat_max_abs_diff': stat,
               'grad_rel_err_vs_grid_barrier_kernels': worst_g[1], 'grad_rel_err_vs_grid_barrier_kernels_tensor': worst_g[0],
               'parity_config': 'fp32 check mode, dropout off, global batch %d of 64x64, DP vs the single-device batch on its default '
                                'dispatch' % Bg}
    import torch.distributed as dist
    dist.barrier()
    return out


def bench_projection_sharded(args, pk, eng_unused, imgs, max_over_ranks, barrier):
    """SURVEY 8e row 1: ONE 3000x512x512 float32 movie split into row bands over the ranks (each rank holds [T, 512/n, 512]),
    band projection without any exchange, all_gather of the 2 x [512/n, 512] maps -> GB/s over the whole movie."""
    import torch
    from deepcalcium.engine.dist import Comm, shard_range, summarize_movie_sharded
    comm = Comm()
    T, H, W = 3000, 512, 512
    first, rows = shard_range(H, comm.world, comm.rank)
    g = torch.Generator(device='cuda'); g.manual_seed(7535 + comm.rank)
    band = torch.rand((T, rows, W), device='cuda', generator=g) * 4096
    for _ in range(3):
        mean, mx = summarize_movie_sharded(band, comm, H)
    barrier()
    n = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        mean, mx = summarize_movie_sharded(band, comm, H)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / n
    # parity: this rank's rows of the gathered maps against torch reductions of its own band (max bit-exact, mean 1e-6)
    ok = bool(torch.equal(mx[first:first + rows], band.amax(0))) and \
        bool(((mean[first:first + rows].double() - band.double().mean(0)).abs() <= 1e-6 * band.double().mean(0).abs()).all())
    t = torch.tensor([1.0 if ok else 0.0], device='cuda')
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MIN)
    nbytes = T * H * W * 4 + 2 * H * W * 4
    del band
    return {'ms_per_movie': ms, 'movies_per_s': 1e3 / ms, 'ranks': comm.world, 'achieved_gbs_aggregate': nbytes / ms / 1e6,
            'frac_of_aggregate_hbm_peak': nbytes / ms / 1e6 / (pk['hbm'] * comm.world), 'parity_ok_all_ranks': bool(t.item() > 0.5),
            'collective': 'all_gather of 2 x %d x %d float32 per rank' % (rows, W)}


def bench_projection(args, pk):
    """BASELINE config C2: mean/max projection of a 3000x512x512 float32 movie resident in HBM."""
    import torch
    from deepcalcium.datasets.nf import summarize_movie_device
    from deepcalcium.engine import ops
    T, H, W = 3000, 512, 512
    g = torch.Generator(device='cuda'); g.manual_seed(7535)
    movie = torch.rand((T, H, W), device='cuda', generator=g) * 4096
    out = (torch.empty(H, W, device='cuda'), torch.empty(H, W, device='cuda'))
    ws = torch.empty(ops.proj_workspace_bytes(T, H, W), dtype=torch.uint8, device='cuda')
    for _ in range(3):
        summarize_movie_device(movie, out=out, workspace=ws)
    torch.cuda.synchronize()
    n = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        summarize_movie_device(movie, out=out, workspace=ws)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    nbytes = T * H * W * 4 + 2 * H * W * 4
    res = {'ms': ms, 'movies_per_s': 1e3 / ms, 'roofline': {'bound': 'hbm', 'achieved': nbytes / ms / 1e6, 'peak': pk['hbm'],
                                                            'unit': 'GB/s', 'frac': nbytes / ms / 1e6 / pk['hbm'],
                                                            'bytes': nbytes, 'note': '3.1 GB input >> L2'}}
    # numpy baseline on a bounded sample (300 frames)
    sub = movie[:300].cpu().numpy()
    t0 = time.perf_counter()
    sub.mean(0, dtype=np.float64); sub.max(0)
    dt = time.perf_counter() - t0
    res['cpu_baseline'] = {'value': sub.nbytes / dt / 1e9, 'unit': 'GB/s', 'cores': 1, 'kind': 'port',
                           'sample': '300 of 3000 frames, numpy mean(float64)+max'}
    # the same movie as int16 frames (the reference's raw TIFF dtype): half the bytes, exact integer sums
    movie16 = movie.to(torch.int16)
    del movie
    for _ in range(3):
        summarize_movie_device(movie16, out=out, workspace=ws)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        summarize_movie_device(movie16, out=out, workspace=ws)
    e1.record()
    torch.cuda.synchronize()
    ms16 = e0.elapsed_time(e1) / n
    nb16 = T * H * W * 2 + 2 * H * W * 4
    res['int16'] = {'ms': ms16, 'movies_per_s': 1e3 / ms16,
                    'roofline': {'bound': 'hbm', 'achieved': nb16 / ms16 / 1e6, 'peak': pk['hbm'], 'unit': 'GB/s',
                                 'frac': nb16 / ms16 / 1e6 / pk['hbm'], 'bytes': nb16}}
    del movie16
    return res


def train_precision(args):
    return 'bf16' if args.precision == 'fp16' else args.precision      # fp16 is inference only


def bench_train(args, pk):
    """BASELINE config C3: 128x128 crops, batch 32, bf16, dice loss, Adam(0.002), dropout on."""
    import torch
    from deepcalcium.engine.graph import GraphSpec, he_normal_weights
    from deepcalcium.engine.unet_engine import UNetEngine
    spec = GraphSpec(32)
    eng = UNetEngine(spec, precision=train_precision(args))
    eng.set_weights_dict(he_normal_weights(spec, seed=7535))
    rng = np.random.default_rng(865)
    B = 32
    xs = [torch.from_numpy(rng.standard_normal((B, 128, 128)).astype(np.float32)).cuda() for _ in range(4)]
    ys = [torch.from_numpy((rng.random((B, 128, 128)) < 0.126).astype(np.uint8)).cuda() for _ in range(4)]
    for i in range(5):
        eng.train_step(xs[i % 4], ys[i % 4], loss='dice_loss', lr=0.002, dropout=True)
    torch.cuda.synchronize()
    n = 20
    l0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        m = eng.train_step(xs[i % 4], ys[i % 4], loss='dice_loss', lr=0.002, dropout=True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    fl = B * spec.flops_train(128, 128)
    res = {'crops_per_s': B * 1e3 / ms, 'ms_per_step': ms, 'batch': B, 'crop': 128, 'loss': 'dice_loss',
           'dtype': train_precision(args), 'final_loss': float(m[0].item()), 'tflops': fl / ms / 1e9, 'frac_of_bf16_peak_burst': fl / ms / 1e9 / pk['tf'],
           'frac_of_bf16_peak_sustained': fl / ms / 1e9 / pk['tf_sus'], 'flops_per_step': fl,
           'gpu_launches_per_step': (eng.launches - l0) // n}
    try:
        res['parity'] = parity_train(train_precision(args), he_normal_weights(spec, seed=7535), xs[0], ys[0])
    except Exception as ex:   # noqa: BLE001
        res['parity'] = {'error': repr(ex)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--precision', default='fp16', choices=['fp16', 'bf16', 'fp32'],
                    help="activation / weight storage of the inference path: fp16 and bf16 run the same tcgen05 kind::f16 MMAs "
                         "(fp32 accumulate) at the same rate; fp16 meets the north star's 1e-2 logit tolerance, bf16 cannot "
                         "(tests/test_gpu_unet.py, DESIGN.md section 4); training extras always run in bf16 (or fp32)")
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the mask and activation the last timed step returned as DIR/mask.npy and DIR/act.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
