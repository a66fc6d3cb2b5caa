"""Which tensor-core kernel every contraction entry point dispatches to.

For each case (shape x dispatch policy x dtype) the table in tests/golden/dispatch_table.json holds, per call, the
dcb_last_kernel() name, the number of kernels the call launched (dcb_launch_count delta) and, for the statistics
entry points, stats_done.  The cases are those of the parity tests in test_gpu_ops.py plus the layers of a 32 x 128^2
training step, so a change to the host dispatch code that moves any of them to another kernel fails here.  After an
intended dispatch change, regenerate the table with DCB_RECORD_DISPATCH=<json file to write> and review its diff."""
import json
import os

import pytest
import torch

import oracle
from test_gpu_ops import CONV_CASES, CONVT_CASES, FUSED_SHAPES, FWD_VARIANTS, WGRAD_VARIANTS

pytestmark = pytest.mark.gpu

TABLE = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'dispatch_table.json')
DT = {'bf16': torch.bfloat16, 'fp16': torch.float16}


def _z(*shape, dtype=torch.bfloat16):
    return torch.zeros(*shape, dtype=dtype, device='cuda')


def _call(nat, fn, *args):
    """[kernel name, launches] of one entry-point call (+ its return value when it has one)"""
    n0 = nat.launch_count()
    r = fn(*args)
    torch.cuda.synchronize()
    row = [nat.last_kernel(), nat.launch_count() - n0]
    return row + [int(r)] if r is not None else row


def _conv_rows(nat, ops):
    rows = {}
    for case in CONV_CASES:
        N, H, W, C0, C1, Cout = case
        Cin = C0 + C1
        for prec, dt in DT.items():
            x0 = _z(N, H, W, C0, dtype=dt)
            x1 = _z(N, H, W, C1, dtype=dt) if C1 else None
            w = _z(9 * Cin * Cout, dtype=dt)
            out = _z(N, H, W, Cout, dtype=dt)
            dy = _z(N, H, W, Cout, dtype=dt)
            dx = _z(N, H, W, Cin, dtype=torch.float32)
            for vname, pol in FWD_VARIANTS:
                with nat.policy(**pol):
                    rows['%s %s %s' % (case, prec, vname)] = [_call(nat, ops.conv3x3_fwd, x0, x1, w, out, None, None, True),
                                                              _call(nat, ops.conv3x3_dgrad, dy, w, dx)]
            if prec == 'bf16':          # the fp16 mode has no gradients
                dW = _z(3, 3, Cin, Cout, dtype=torch.float32)
                for vname, pol in WGRAD_VARIANTS:
                    with nat.policy(**pol):
                        ws = _z(max(16, ops.conv3x3_wgrad_workspace_bytes(dt, N, H, W, Cin, Cout)), dtype=torch.uint8)
                        rows['%s %s wgrad %s' % (case, prec, vname)] = [_call(nat, ops.conv3x3_wgrad, x0, x1, dy, dW, ws)]
    return rows


def _fused_rows(nat, ops):
    rows = {}
    for shape in FUSED_SHAPES:
        N, H, W, Cin, Cout = shape
        for prec, dt in DT.items():
            x = _z(N, H, W, Cin, dtype=dt)
            w = _z(9 * Cin * Cout, dtype=dt)
            y = _z(N, H, W, Cout, dtype=dt)
            pool = _z(N, H // 2, W // 2, Cout, dtype=dt)
            hk = _z(Cout, 2, dtype=torch.float32)
            hb = _z(2, dtype=torch.float32)
            logit = _z(N, H, W, dtype=torch.float32)
            prob = _z(N, H, W, dtype=torch.float32)
            for pair in (1, 0):
                with nat.policy(pair=pair):
                    pooled = _call(nat, lambda: ops.conv3x3_fwd_fused(x, None, w, y, None, None, True, pool_out=pool))
                    head = _call(nat, lambda: ops.conv3x3_fwd_fused(x, None, w, y, None, None, True, head_kernel=hk, head_bias=hb,
                                                                    logit=logit, prob=prob, need_y=False))
                    rows['%s %s pair %d' % (shape, prec, pair)] = [pooled, head]
    return rows


def _stats_rows(nat, ops):
    """dcb_conv3x3_fwd_stats / dcb_convT2x2_fwd_stats at the layers of a 32 x 128^2 training step (nb_filters_base 32;
    decoder convs read [upsampled, skip] as two sources)"""
    rows = {}
    N, S = 32, 128
    level = {'enc0': 0, 'enc1': 1, 'enc2': 2, 'enc3': 3, 'bot': 4, 'dec3': 3, 'dec2': 2, 'dec1': 1, 'dec0': 0}
    for name, kind, cin, cout in oracle.UNetSpec(nb_filters_base=32).blocks():
        if kind == 'head' or cin == 1:
            continue
        for fused_bn in (2, 3):
            with nat.policy(fused_bn=fused_bn):
                sums = _z(2 * cout, dtype=torch.int64)
                if kind == 'up':
                    h = S >> (int(name[2:]) + 1)
                    call = _call(nat, ops.convT2x2_fwd_stats, _z(N, h, h, cin), _z(4 * cin * cout), _z(N, 2 * h, 2 * h, cout), sums)
                else:
                    H = S >> level[name[:-1]]
                    two = name.startswith('dec') and name.endswith('a')
                    C0 = cin // 2 if two else cin
                    call = _call(nat, ops.conv3x3_fwd_stats, _z(N, H, H, C0), _z(N, H, H, cin - C0) if two else None,
                                 _z(9 * cin * cout), _z(N, H, H, cout), sums)
                rows['%s fused_bn %d' % (name, fused_bn)] = [call]
    return rows


def _convT_rows(nat, ops):
    rows = {}
    for case in CONVT_CASES:
        N, h, w_, Cin, Cout = case
        for prec, dt in DT.items():
            x = _z(N, h, w_, Cin, dtype=dt)
            wf = _z(4 * Cin * Cout, dtype=dt)
            out = _z(N, 2 * h, 2 * w_, Cout, dtype=dt)
            dy = _z(N, 2 * h, 2 * w_, Cout, dtype=dt)
            dx = _z(N, h, w_, Cin, dtype=torch.float32)
            dW = _z(2, 2, Cout, Cin, dtype=torch.float32)
            for tma_store in (1, 0):
                with nat.policy(tma_store=tma_store):
                    calls = [_call(nat, ops.convT2x2_fwd, x, wf, out, None, None, False),
                             _call(nat, ops.convT2x2_dgrad, dy, wf, dx)]
                    if prec == 'bf16':
                        ws = _z(max(16, ops.convT2x2_wgrad_workspace_bytes(dt, N, h, w_, Cin, Cout)), dtype=torch.uint8)
                        calls.append(_call(nat, ops.convT2x2_wgrad, x, dy, dW, ws))
                    rows['%s %s tma_store %d' % (case, prec, tma_store)] = calls
    return rows


GROUPS = {'conv3x3': _conv_rows, 'fused': _fused_rows, 'stats': _stats_rows, 'convT2x2': _convT_rows}


@pytest.mark.parametrize('group', list(GROUPS))
def test_dispatch_table(cuda, group):
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    nat.reset_policy()
    got = GROUPS[group](nat, ops)
    record = os.environ.get('DCB_RECORD_DISPATCH')
    if record:
        table = json.load(open(record)) if os.path.exists(record) else {}
        table[group] = got
        with open(record, 'w') as f:
            json.dump(table, f, indent=0, sort_keys=True)
        return
    want = json.load(open(TABLE))[group]
    assert sorted(got) == sorted(want)
    diff = ['%s: %s, recorded %s' % (k, got[k], want[k]) for k in sorted(want) if got[k] != want[k]]
    assert not diff, '%d of %d cases dispatch differently:\n%s' % (len(diff), len(want), '\n'.join(diff[:40]))
