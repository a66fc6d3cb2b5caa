"""Dataset preparation of the reference (deepcalcium/datasets/nf.py), hot-path part only:
the per-pixel temporal mean / max projection of a movie (nf.py:115-130; twin loop at
examples/neurons/unet2ds_sj.py:67-85) runs as one streaming CUDA kernel.

``summarize_movie`` is the projection as a function (movie in, (mean, max) out);
``make_dataset`` writes the reference's dataset schema (series/mean, series/max, masks/raw,
masks/max, attr name, nf.py:39-44): ``*.hdf5`` / ``*.h5`` paths in the reference's HDF5 layout (through h5py when it
is importable, else the pure-Python classic-format writer utils/hdf5_lite.py), other paths as an ``.npz`` container.
Neurofinder download / unzip / TIFF decode (nf.py:73-97, 126-127) are out of scope (no network).
"""
import logging
import os

import numpy as np

from ..utils.runtime import funcname

NEUROFINDER_NAMES = sorted([
    'neurofinder.00.00', 'neurofinder.00.01', 'neurofinder.00.02', 'neurofinder.00.03', 'neurofinder.00.04',
    'neurofinder.00.05', 'neurofinder.00.06', 'neurofinder.00.07', 'neurofinder.00.08', 'neurofinder.00.09',
    'neurofinder.00.10', 'neurofinder.00.11', 'neurofinder.01.00', 'neurofinder.01.01', 'neurofinder.02.00',
    'neurofinder.02.01', 'neurofinder.03.00', 'neurofinder.04.00', 'neurofinder.04.01',
    'neurofinder.00.00.test', 'neurofinder.00.01.test', 'neurofinder.01.00.test', 'neurofinder.01.01.test',
    'neurofinder.02.00.test', 'neurofinder.02.01.test', 'neurofinder.03.00.test', 'neurofinder.04.00.test',
    'neurofinder.04.01.test'])


def summarize_movie_device(movie_dev, floor_max_at_zero=False, variant=-1, t_splits=0, out=None, workspace=None):
    """movie_dev: float32 or int16 CUDA tensor [T,H,W].  Returns (mean, max) float32 CUDA tensors [H,W]."""
    import torch
    from ..engine import ops
    if movie_dev.dim() != 3:
        raise ValueError('movie must be [T,H,W], got shape %s' % (tuple(movie_dev.shape),))
    if movie_dev.shape[0] == 0:
        raise ValueError('movie has no frames')
    if movie_dev.dtype not in (torch.float32, torch.int16) or not movie_dev.is_cuda:
        raise TypeError('summarize_movie_device needs a float32 or int16 CUDA tensor')
    movie_dev = movie_dev.contiguous()
    T, H, W = movie_dev.shape
    if out is None:
        out = (torch.empty(H, W, dtype=torch.float32, device=movie_dev.device),
               torch.empty(H, W, dtype=torch.float32, device=movie_dev.device))
    if workspace is None:
        workspace = torch.empty(ops.proj_workspace_bytes(T, H, W), dtype=torch.uint8, device=movie_dev.device)
    ops.proj_mean_max(movie_dev, out[0], out[1], workspace, floor_max_at_zero, variant, t_splits)
    return out


def summarize_masks_device(masks_dev):
    """masks_dev: int8, uint8 or bool CUDA tensor [n,H,W], one plane per neuron (a neuron owns the pixels where its plane
    == 1).  Returns the truth mask of _summarize_mask (unet_2d_summary.py:244-291) as a uint8 CUDA tensor [H,W]: pixels
    owned by one neuron, minus every 3x3 neighbourhood the reference's walk finds touching two neurons."""
    import torch
    from ..engine import ops
    if masks_dev.dim() != 3:
        raise ValueError('masks must be [n,H,W], got shape %s' % (tuple(masks_dev.shape),))
    if masks_dev.dtype not in (torch.int8, torch.uint8, torch.bool) or not masks_dev.is_cuda:
        raise TypeError('summarize_masks_device needs an int8, uint8 or bool CUDA tensor, got %s on %s'
                        % (masks_dev.dtype, masks_dev.device))
    masks_dev = masks_dev.contiguous()
    n, H, W = masks_dev.shape
    with torch.cuda.device(masks_dev.device):
        out = torch.empty(H, W, dtype=torch.uint8, device=masks_dev.device)
        ws = torch.empty(ops.mask_summary_workspace_bytes(n, H, W), dtype=torch.uint8, device=masks_dev.device)
        ops.mask_summary(masks_dev, out, ws)
    return out


def summarize_movie(movie, floor_max_at_zero=False):
    """Mean / max projection of a [T,H,W] movie given as a numpy array (any real dtype; the
    reference's TIFF frames are int16, nf.py:121) -> (mean float32 [H,W], max float32 [H,W]).
    ``floor_max_at_zero=True`` reproduces the reference's zero-initialised running max (nf.py:125)."""
    import torch
    from .. import _native as nat
    nat.require_cuda()
    movie = np.asarray(movie)
    if movie.ndim != 3:
        raise ValueError('movie must be [T,H,W], got shape %s' % (movie.shape,))
    # int16 frames (the reference's TIFFs) go to the device as they are: half the PCIe and HBM bytes, exact sums
    host = np.ascontiguousarray(movie) if movie.dtype == np.int16 else np.ascontiguousarray(movie, dtype=np.float32)
    dev = torch.from_numpy(host).cuda()
    mean, mx = summarize_movie_device(dev, floor_max_at_zero)
    return mean.cpu().numpy(), mx.cpu().numpy()


# ------------------------------------------------------------------ dataset container
def _is_hdf5(path):
    return path.endswith(('.hdf5', '.h5'))


def _h5():
    """h5py when it is importable, else the pure-Python classic-format reader / writer (utils/hdf5_lite.py)"""
    try:
        import h5py
        return h5py
    except ImportError:
        from ..utils import hdf5_lite
        return hdf5_lite


def open_dataset(path, keys=None):
    """Read a dataset file into a dict {'name', 'series/mean', 'series/max', 'masks/raw', ...}: the reference's HDF5
    schema (datasets/nf.py:39-44; ``series/raw``, the movie itself, is not loaded) or the .npz container.
    ``keys``: read only these arrays (e.g. ``('masks/raw',)``; missing ones are left out); 'name' is always there."""
    want = None if keys is None else set(keys)
    if _is_hdf5(path):
        out = {}
        with _h5().File(path, 'r') as fp:
            name = fp.attrs['name']
            out['name'] = name.decode('utf8') if isinstance(name, bytes) else str(name)
            for grp in ('series', 'masks'):
                if grp in fp:
                    for k in fp[grp].keys():
                        key = '%s/%s' % (grp, k)
                        if (k != 'raw' or grp == 'masks') and (want is None or key in want):
                            out[key] = np.asarray(fp[grp][k][...])
        return out
    with np.load(path, allow_pickle=False) as z:
        out = {k.replace('__', '/'): z[k] for k in z.files
               if want is None or k == 'name' or k.replace('__', '/') in want}
    out['name'] = str(out['name'])
    return out


def make_dataset(path, name, movie=None, mean=None, mx=None, masks=None):
    """Write the reference's dataset schema.  Either ``movie`` ([T,H,W], projected on the GPU) or
    precomputed ``mean``/``mx`` must be given.  series/mean is stored as float16 and series/max as
    int16 like the reference (nf.py:122-125); masks/raw int8 [n,H,W], masks/max int8 [H,W]."""
    if movie is not None:
        mean, mx = summarize_movie(movie, floor_max_at_zero=True)
    d = {'name': np.asarray(name), 'series__mean': np.asarray(mean).astype(np.float16),
         # HDF5's integer conversion saturates (the reference assigns into an int16 dataset, nf.py:124,130)
         'series__max': np.clip(np.asarray(mx), -32768, 32767).astype(np.int16)}
    if masks is not None:
        masks = np.asarray(masks).astype(np.int8)
        d['masks__raw'] = masks
        d['masks__max'] = masks.max(axis=0)
    if _is_hdf5(path):
        with _h5().File(path, 'w') as fp:
            fp.attrs['name'] = name
            for k, v in d.items():
                if k != 'name':
                    fp.create_dataset(k.replace('__', '/'), data=v)
    else:
        np.savez(path, **d)
    return path


def nf_load_hdf5(names, datasets_dir=None):
    """Reference entry point (nf.py:37).  Downloading Neurofinder needs network access and TIFF /
    HDF5 libraries that are outside this build's scope; datasets that were already prepared
    (``<datasets_dir>/<name>/dataset.hdf5`` or ``dataset.npz``) are returned, otherwise an error
    says what is missing."""
    logger = logging.getLogger(funcname())
    if datasets_dir is None:
        from ..utils.config import DATASETS_DIR
        datasets_dir = '%s/neurons_nf' % DATASETS_DIR
    if isinstance(names, str) and names.lower() == 'all':
        dataset_names = NEUROFINDER_NAMES
    elif isinstance(names, str) and names.lower() == 'all_train':
        dataset_names = sorted([n for n in NEUROFINDER_NAMES if '.test' not in n])
    elif isinstance(names, str) and names.lower() == 'all_test':
        dataset_names = sorted([n for n in NEUROFINDER_NAMES if '.test' in n])
    elif isinstance(names, str):
        dataset_names = names.split(',')
    else:
        dataset_names = names
    paths = []
    for name in dataset_names:
        for fn in ('dataset.hdf5', 'dataset.npz'):
            p = '%s/%s/%s' % (datasets_dir, name, fn)
            if os.path.exists(p):
                logger.info('%s already prepared.' % p)
                paths.append(p)
                break
        else:
            raise FileNotFoundError('%s/%s: no prepared dataset; download + TIFF decode (nf.py:73-127) are out '
                                    'of scope here - build one with make_dataset()' % (datasets_dir, name))
    return paths


# ------------------------------------------------------------------------------------------------- ingest (N4)
def _read_tiff_frame(path):
    """One 16-bit greyscale TIFF frame -> (int16 array, bias).  Neurofinder TIFFs are uint16; the reference computes
    series/mean and series/max from the UNWRAPPED pixel values (nf.py:129-130 work on `img`, not on the int16 copy),
    so unsigned frames are shifted into the int16 range (value - 32768 = bits ^ 0x8000) for the exact integer kernel and
    the bias is added back after the projection.  Signed frames pass through with bias 0."""
    from PIL import Image
    with Image.open(path) as im:
        a = np.asarray(im)
    if a.ndim != 2:
        raise ValueError('%s: expected a single greyscale frame, got shape %s' % (path, a.shape))
    if a.dtype == np.uint16:
        return (a ^ np.uint16(0x8000)).view(np.int16), 32768
    if a.dtype == np.uint8 or a.dtype == np.int16 or a.dtype == np.int8:
        return a.astype(np.int16, copy=False), 0
    if np.issubdtype(a.dtype, np.integer) and a.min() >= -32768 and a.max() <= 32767:
        return a.astype(np.int16), 0
    raise ValueError('%s: pixel type %s does not fit the 16-bit ingest path' % (path, a.dtype))


def summarize_tiff_dir(images_dir, chunk=64, floor_max_at_zero=True, pattern=('*.tiff', '*.tif')):
    """The reference's ingest loop (datasets/nf.py:115-130) without materialising the movie: the TIFF frames of
    `images_dir` (sorted by name) are decoded into a pinned int16 double buffer `chunk` frames at a time, copied to the
    GPU on a side stream and folded into the device-resident running sum (exact int64) / max (dcb_proj_accum_i16) while
    the host decodes the next chunk.  Returns (mean float32 [H,W], max float32 [H,W], number of frames).
    floor_max_at_zero=True reproduces the reference's zero-initialised running max (nf.py:125)."""
    import glob
    import torch
    from .. import _native as nat
    from ..engine import ops
    nat.require_cuda()
    paths = sorted(p for pat in pattern for p in glob.glob(os.path.join(images_dir, pat)))
    if not paths:
        raise ValueError('no TIFF frames in %s' % images_dir)
    first, bias = _read_tiff_frame(paths[0])
    H, W = first.shape
    dev = torch.device('cuda', torch.cuda.current_device())
    hbuf = [torch.empty(chunk, H, W, dtype=torch.int16).pin_memory() for _ in range(2)]
    dbuf = [torch.empty(chunk, H, W, dtype=torch.int16, device=dev) for _ in range(2)]
    done = [torch.cuda.Event(), torch.cuda.Event()]
    ssum = torch.zeros(H, W, dtype=torch.int64, device=dev)
    smax = torch.full((H, W), -2 ** 31, dtype=torch.int32, device=dev)
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream(dev)
    for c, i0 in enumerate(range(0, len(paths), chunk)):
        k = c % 2
        done[k].synchronize()                                # chunk c-2 has been consumed: its buffers are free
        n = min(chunk, len(paths) - i0)
        hv = hbuf[k].numpy()
        for j in range(n):
            fr, fb = (first, bias) if i0 + j == 0 else _read_tiff_frame(paths[i0 + j])
            if fr.shape != (H, W) or fb != bias:
                raise ValueError('%s: frame shape / pixel type %s differs from the first frame %s' % (paths[i0 + j], fr.shape, (H, W)))
            hv[j] = fr
        with torch.cuda.stream(copy_stream):
            dbuf[k][:n].copy_(hbuf[k][:n], non_blocking=True)
            ready = torch.cuda.Event(); ready.record(copy_stream)
        main.wait_event(ready)
        ops.proj_accum_i16(dbuf[k][:n], ssum, smax)
        done[k].record(main)
    mean = torch.empty(H, W, dtype=torch.float32, device=dev)
    mx = torch.empty(H, W, dtype=torch.float32, device=dev)
    # unsigned frames were shifted by -32768: the device restores the bias in exact integer arithmetic
    ops.proj_accum_finalize(ssum, smax, len(paths), mean, mx, floor_max_at_zero, bias)
    return mean.cpu().numpy(), mx.cpu().numpy(), len(paths)


def nf_ingest(name, datasets_dir, out_path=None, chunk=64):
    """nf.py:104-148 for one already-downloaded neurofinder dataset directory `<datasets_dir>/<name>` (images/*.tiff and,
    for training sets, regions/regions.json): summary images through the streaming GPU projection, masks from the region
    coordinates, written as the `.npz` container of make_dataset.  (Download / unzip stay out of scope: no network.)"""
    import json
    root = os.path.join(datasets_dir, name)
    mean, mx, T = summarize_tiff_dir(os.path.join(root, 'images'), chunk=chunk)
    masks = None
    rj = os.path.join(root, 'regions', 'regions.json')
    if '.test' not in name and os.path.exists(rj):
        with open(rj) as fp:
            regions = json.load(fp)
        masks = np.zeros((len(regions),) + mean.shape, dtype=np.int8)
        for idx, r in enumerate(regions):
            yy, xx = [c[0] for c in r['coordinates']], [c[1] for c in r['coordinates']]
            masks[idx, yy, xx] = 1
    out_path = out_path or os.path.join(root, 'dataset.hdf5')
    return make_dataset(out_path, name, mean=mean, mx=mx, masks=masks)


# ------------------------------------------------------------------------------------------------- scoring (N3)
# datasets/nf.py:153-229 of the reference scores a predicted mask by converting both masks to connected regions
# (skimage.measure.label, default = 8-connectivity in 2-D) and calling `neurofinder.centers` / `neurofinder.shapes`
# (neurofinder==1.1.1 on regional==1.1.2, requirements.txt).  Neither package is importable here, so their published
# algorithm is restated (PARITY UNPINNED, like the rest of the oracle-backed path):
#   match(a, b, threshold): for every region s of a, in order: the nearest REMAINING region of b by centre distance
#       (centre = mean of the pixel coordinates); it is taken (and removed from b) if that distance < threshold.
#   centers(a, b, threshold=5) -> (recall, precision) = (#matched pairs with distance < threshold) / len(a), / len(b)
#   shapes(a, b, threshold=5)  -> (inclusion, exclusion) = mean over the matched pairs of
#       (|s_a & s_b| / |s_a|, |s_a & s_b| / |s_b|)  (regional.one.overlap(method='rates')); (0, 0) without pairs.

def _label_regions(m):
    """Connected components of a binary mask as a list of [k, 2] (row, col) coordinate arrays, 8-connected, numbered
    in raster order of their first pixel (skimage.measure.label's numbering)."""
    from scipy import ndimage
    lbl, n = ndimage.label(np.asarray(m) != 0, structure=np.ones((3, 3), dtype=bool))
    if n == 0:
        return []
    order = np.argsort(lbl.ravel(), kind='stable')
    flat = lbl.ravel()[order]
    starts = np.searchsorted(flat, np.arange(1, n + 2))
    rows, cols = np.unravel_index(order, lbl.shape)
    return [np.stack([rows[starts[k]:starts[k + 1]], cols[starts[k]:starts[k + 1]]], axis=1) for k in range(n)]


def _match_regions(a, b, threshold):
    """neurofinder.match: index into b (or None) for every region of a."""
    ca = [r.mean(axis=0) for r in a]
    targets = np.array([r.mean(axis=0) for r in b], dtype=np.float64).reshape(len(b), 2)
    target_inds = list(range(len(b)))
    out = []
    for c in ca:
        hit = None
        if len(target_inds):
            d = np.sqrt(((targets - c[np.newaxis]) ** 2).sum(axis=1))
            k = int(np.argmin(d))
            if d[k] < threshold:
                hit = target_inds[k]
                targets = np.delete(targets, k, axis=0)
                del target_inds[k]
        out.append(hit)
    return out


def _overlaps(a, b, match):
    """|s_a & s_b| of every truth region and its matched prediction region (0 without a match)"""
    out = []
    for ra, ib in zip(a, match):
        if ib < 0:
            out.append(0)
            continue
        sa = set(map(tuple, ra.tolist()))
        out.append(sum(1 for xy in map(tuple, b[ib].tolist()) if xy in sa))
    return out


def _match_stats(a, b, threshold):
    """(match index or -1 per truth region, truth sizes, prediction sizes, overlaps) of two region lists"""
    match = [-1 if ib is None else ib for ib in _match_regions(a, b, threshold)]
    return match, [len(r) for r in a], [len(r) for r in b], _overlaps(a, b, match)


def nf_scores_from_matches(na, nb, match, size_a, size_b, nhit):
    """The float arithmetic of neurofinder.centers / shapes and the combined score, from a matching: na truth and nb
    prediction regions, match[k] = index of the prediction region matched to truth region k or -1, size_a / size_b the
    region pixel counts, nhit[k] the overlap of truth region k with its match.  -> (prec, reca, incl, excl, comb).
    Every matched pair is closer than the threshold (the matching only takes such pairs), so it counts for centers.
    Host and device scoring both end here, so their five numbers come from the same expressions."""
    match = np.asarray(match, dtype=np.int64).reshape(-1)
    hit = match >= 0
    n = int(np.count_nonzero(hit))
    with np.errstate(divide='ignore', invalid='ignore'):
        r, p = np.float64(n) / np.float64(na), np.float64(n) / np.float64(nb)
    if n:
        nh = np.asarray(nhit, dtype=np.float64).reshape(-1)[hit]
        sa = np.asarray(size_a, dtype=np.float64).reshape(-1)[hit]
        sb = np.asarray(size_b, dtype=np.float64).reshape(-1)[match[hit]]
        rates = np.stack([nh / sa, nh / sb], axis=1)
        i, e = (float(v) for v in rates.mean(axis=0))
    else:
        i, e = 0.0, 0.0
    with np.errstate(divide='ignore', invalid='ignore'):
        f1 = np.float64(2.) * (r * p) / (r + p)
    return (float(p), float(r), float(i), float(e), float(f1))


def nf_centers(a, b, threshold=5):
    """neurofinder.centers on two region lists -> (recall, precision)."""
    p, r = nf_scores_from_matches(len(a), len(b), *_match_stats(a, b, threshold))[:2]
    return np.float64(r), np.float64(p)


def nf_shapes(a, b, threshold=5):
    """neurofinder.shapes on two region lists -> (inclusion, exclusion)."""
    return nf_scores_from_matches(len(a), len(b), *_match_stats(a, b, threshold))[2:4]


def nf_mask_metrics(m, mp):
    """datasets/nf.py:153-174: precision, recall, inclusion, exclusion and combined (F1) score of a predicted mask.
    Single 2-D masks, overlapping neurons are not accounted for (as in the reference)."""
    mp = np.asarray(mp)
    if np.sum(mp.round()) == 0:
        return 0., 0., 0., 0., 0.
    a, b = _label_regions(m), _label_regions(mp)
    return nf_scores_from_matches(len(a), len(b), *_match_stats(a, b, 5))


# device scoring: one table row per image (ops.nf_score); kind 0 = uint8 nonzero, 1 / 2 = fp32 / fp64 round(p) != 0
_SCORE_KINDS = {'torch.uint8': 0, 'torch.bool': 0, 'torch.float32': 1, 'torch.float64': 2}


def _tensor_row(t):
    kind = _SCORE_KINDS.get(str(t.dtype))
    if not t.is_cuda or t.dim() != 2 or kind is None:
        raise TypeError('nf_mask_metrics_device takes 2-D CUDA masks of dtype uint8, bool, float32 or float64, got %s %s %s'
                        % (t.device, t.dtype, tuple(t.shape)))
    return [t.data_ptr(), t.shape[0], t.shape[1], t.stride(0), t.stride(1), kind, 0, 0]


def nf_metrics_from_table(h_desc, device):
    """Score the (truth, prediction) image pairs of an int64 table [2 n, 8] (rows as in ops.nf_score; the images must stay
    alive until this returns) -> n tuples (prec, reca, incl, excl, comb)."""
    import torch
    from ..engine import ops
    h_desc = np.ascontiguousarray(h_desc, dtype=np.int64)
    n = h_desc.shape[0] // 2
    if n == 0:
        return []
    nbytes, cap = ops.nf_score_workspace_bytes(h_desc)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    info = torch.empty(max(cap, 1), 3, dtype=torch.int32, device=device)
    base = torch.empty(2 * n + 1, dtype=torch.int32, device=device)
    ops.nf_score(torch.from_numpy(h_desc).to(device), h_desc, base, info, ws)
    hbase = base.cpu().numpy().astype(np.int64)
    hinfo = info[:int(hbase[-1])].cpu().numpy()
    out = []
    for i in range(n):
        a0, a1, b1 = hbase[2 * i], hbase[2 * i + 1], hbase[2 * i + 2]
        if b1 == a1:                     # no predicted region: nf_mask_metrics' early exit
            out.append((0., 0., 0., 0., 0.))
            continue
        ta = hinfo[a0:a1]
        out.append(nf_scores_from_matches(a1 - a0, b1 - a1, ta[:, 1], ta[:, 0], hinfo[a1:b1, 0], ta[:, 2]))
    return out


def nf_mask_metrics_device(pairs):
    """nf_mask_metrics for a batch of (truth, prediction) masks that are already on the GPU: 2-D CUDA tensors with values
    in {0, 1} (uint8, bool, float32 or float64; any strides, shapes may differ between pairs but not within one).
    Labelling, region statistics, the centre matching and the overlaps run in one device call (ops.nf_score); only the
    per-region integers come back.  Returns one (prec, reca, incl, excl, comb) tuple per pair, equal bit for bit to
    nf_mask_metrics(truth.cpu(), pred.cpu()), NaN included."""
    pairs = list(pairs)
    if not pairs:
        return []
    rows = []
    for t, p in pairs:
        if tuple(t.shape) != tuple(p.shape):
            raise ValueError('truth %s and prediction %s differ in shape' % (tuple(t.shape), tuple(p.shape)))
        rows += [_tensor_row(t), _tensor_row(p)]
    return nf_metrics_from_table(np.asarray(rows, dtype=np.int64), pairs[0][0].device)


def nf_submit(Mp, names, json_path):
    """datasets/nf.py:177-217: Neurofinder submission JSON.  Kept bug-compatible with the reference: the region loop is
    `range(1, max_label)`, i.e. the LAST connected component of every mask is not written."""
    import json
    logger = logging.getLogger(funcname())
    submission = []
    for mp, name in zip(Mp, names):
        if name.startswith('neurofinder.'):
            name = '.'.join(name.split('.')[1:])
        regs = _label_regions(mp)
        if len(regs) == 0:
            regions = [{'coordinates': [[[0, 0]]]}]
        else:
            regions = [{'coordinates': [[int(y), int(x)] for y, x in r.tolist()]} for r in regs[:len(regs) - 1]]
        submission.append({'dataset': name, 'regions': regions})
    with open(json_path, 'w') as fp:
        json.dump(submission, fp)
    logger.info('Saved submission to %s.' % json_path)
