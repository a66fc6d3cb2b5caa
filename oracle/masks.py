"""Host reference of the truth-mask summary (deepcalcium/models/neurons/unet_2d_summary.py:244-291, _summarize_mask).

This is the body ``_summarize_mask`` had before the summary moved to the device (dcb_mask_summary), kept verbatim as
the yardstick the device result must equal bit for bit.
"""
import numpy as np


def summarize_mask_array(msks):
    """masks [n, H, W] -> float64 [H, W]: flatten the per-neuron masks; drop pixels claimed by more than one
    neuron, then drop any 3x3 neighbourhood that still touches two different neurons (same visiting
    order as the reference: first-seen order of the (y,x) keys)."""
    zz, yy, xx = np.where(msks == 1)
    owner = {}
    for z, y, x in zip(zz.tolist(), yy.tolist(), xx.tolist()):
        owner.setdefault((y, x), []).append(z)
    for k in [k for k, v in owner.items() if len(v) > 1]:
        del owner[k]
    for (y, x) in list(owner.keys()):
        nbrs = [(y - 1, x), (y + 1, x), (y, x - 1), (y, x + 1), (y + 1, x + 1), (y - 1, x - 1), (y + 1, x - 1),
                (y - 1, x + 1), (y, x)]
        nbrs = [k for k in nbrs if k in owner]
        if len(set(owner[k][0] for k in nbrs)) > 1:
            for k in nbrs:
                del owner[k]
    summ = np.zeros(msks.shape[1:])
    if owner:
        ys, xs = zip(*owner.keys())
        summ[list(ys), list(xs)] = 1.
    return summ


def summarize_mask(dspath):
    """the host _summarize_mask plugin: masks/raw of a dataset file -> float64 [H, W]"""
    from deepcalcium.datasets.nf import open_dataset
    return summarize_mask_array(open_dataset(dspath)['masks/raw'])
