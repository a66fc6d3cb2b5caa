"""Multi-GPU partitioning of the hot path (one process per GPU, torch.distributed for the plumbing;
NCCL over NVLink on the GPU box, gloo in the CPU tests).  New functionality - the reference is
single-device - specified in SURVEY.md section 8e:

  * independent units (movies, images, windows): ``shard_range`` splits them, no collective;
  * one image's 8 TTA transforms over n ranks (BASELINE config C4): transform k -> rank owning
    ``shard_range(8, n, r)``; probability maps are gathered to rank 0 and combined in the fixed
    order 0..7, so the mask is bit-identical to the 1-GPU result;
  * data-parallel training (C5): rank r trains on crops ``shard_range(B, n, r)``; BatchNorm batch
    statistics, the loss sums and the gradients are all-reduced (sum) so every rank applies the
    single-device update of the whole global batch.
"""
import torch
import torch.distributed as dist


def shard_range(n_items, world, rank):
    """Contiguous balanced split: returns (first, count) of rank's share of n_items."""
    if not (0 <= rank < world):
        raise ValueError('rank %d outside world %d' % (rank, world))
    base, rem = divmod(n_items, world)
    first = rank * base + min(rank, rem)
    return first, base + (1 if rank < rem else 0)


class Comm(object):
    """The three collectives the path needs.  A Comm of world 1 is a no-op."""

    def __init__(self, group=None):
        self.group = group
        self.enabled = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(group) if self.enabled else 1
        self.rank = dist.get_rank(group) if self.enabled else 0

    def allreduce_sum(self, t):
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t

    def broadcast(self, t, src=0):
        if self.world > 1:
            dist.broadcast(t, src=src, group=self.group)
        return t

    def all_gather_rows(self, t, counts):
        """every rank receives every rank's [K, rows_r, W] tensor (rows_r = counts[r], may differ by one)"""
        pad = max(counts)
        buf = t
        if t.shape[1] < pad:
            buf = torch.zeros((t.shape[0], pad) + tuple(t.shape[2:]), dtype=t.dtype, device=t.device)
            buf[:, :t.shape[1]] = t
        out = [torch.empty_like(buf) for _ in range(self.world)]
        dist.all_gather(out, buf.contiguous(), group=self.group)
        return [o[:, :c] for o, c in zip(out, counts)]

    def gather_to_root(self, t, counts=None):
        """Rank 0 receives every rank's tensor (in rank order) and returns them as a list; other
        ranks return None.  ``counts``: leading-dimension size per rank when shards are uneven."""
        if self.world == 1:
            return [t]
        if counts is None:
            counts = [t.shape[0]] * self.world
        # all_gather keeps the call symmetric (gather is not implemented by every backend/version)
        pad = max(counts)
        buf = t
        if t.shape[0] < pad:
            buf = torch.zeros((pad,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
            buf[:t.shape[0]] = t
        out = [torch.empty_like(buf) for _ in range(self.world)]
        dist.all_gather(out, buf.contiguous(), group=self.group)
        if self.rank != 0:
            return None
        return [o[:c] for o, c in zip(out, counts)]


def predict_tta_sharded(engine, summ_dev, comm, window=512, threshold=0.5, shape=None):
    """One summary image, its 8 TTA transforms sharded over comm.world ranks (1, 2, 4 or 8).  Rank 0 passes the image,
    the other ranks may pass ``summ_dev=None`` and ``shape=(hs, ws)`` (an image given on another rank is only used for its
    shape: the pixels come from rank 0 over NVLink).  Returns (mask, act) device tensors on rank 0, (None, None) elsewhere."""
    if comm.world == 1:
        return engine.predict_tta(summ_dev, window=window, augmentation=True, threshold=threshold)
    st = getattr(engine, '_sharded_tta', None)
    if st is None or st.comm is not comm or st.S != window:
        st = ShardedTTA(engine, comm, window)
        engine._sharded_tta = st
    hs, ws = shape if shape is not None else summ_dev.shape
    return st.predict(summ_dev if comm.rank == 0 else None, hs, ws, threshold)


def summarize_movie_sharded(band, comm, H, floor_max_at_zero=False, project_fn=None):
    """Projection of ONE movie split into row bands over the ranks (SURVEY 8e, row 1; reference loop: datasets/nf.py:126-130).
    The reduction is per pixel, so rank r projects its band ``movie[:, first:first+rows, :]`` with
    ``(first, rows) = shard_range(H, world, r)`` without any exchange; the two [rows, W] float32 maps are then
    all-gathered (2 x 4 x H x W / world bytes per rank) so every rank holds the full (mean, max) images.
    ``band``: [T, rows, W] tensor on this rank's device.  ``project_fn(band, floor_max_at_zero) -> (mean, max)`` defaults
    to the CUDA kernel (deepcalcium.datasets.nf.summarize_movie_device); the CPU tests of the host logic inject one."""
    if project_fn is None:
        from ..datasets.nf import summarize_movie_device
        project_fn = summarize_movie_device
    world, rank = comm.world, comm.rank
    first, rows = shard_range(H, world, rank)
    if band.dim() != 3 or band.shape[1] != rows:
        raise ValueError('rank %d of %d holds rows [%d, %d) of %d: expected a [T, %d, W] band, got %s'
                         % (rank, world, first, first + rows, H, rows, tuple(band.shape)))
    mean, mx = project_fn(band, floor_max_at_zero)
    if world == 1:
        return mean, mx
    both = torch.stack([mean, mx], dim=0)                         # [2, rows, W]
    counts = [shard_range(H, world, r)[1] for r in range(world)]
    parts = comm.all_gather_rows(both, counts)                    # list over ranks of [2, rows_r, W]
    full = torch.cat(parts, dim=1)
    return full[0].contiguous(), full[1].contiguous()


# ------------------------------------------------------------------------------------------ peer-mapped memory
class RawTensor(object):
    """A device buffer that torch does not own (a dcb_peer_alloc'ed buffer or a peer's buffer mapped into this process),
    with just enough of the tensor surface for the C-ABI wrappers in ``ops`` (data_ptr / shape / dtype)."""

    def __init__(self, addr, shape, dtype):
        self.addr, self.shape, self.dtype = int(addr), tuple(int(v) for v in shape), dtype
        self.is_cuda = True

    def data_ptr(self):
        return self.addr

    def is_contiguous(self):
        return True

    def dim(self):
        return len(self.shape)

    def numel(self):
        n = 1
        for v in self.shape:
            n *= v
        return n

    def element_size(self):
        return torch.empty(0, dtype=self.dtype).element_size()


class PeerGroup(object):
    """Peer-mapped buffers over the ranks of one NVSwitch box: ``alloc(nbytes)`` is a collective that returns the list of
    per-rank device addresses of a zero-filled buffer of that size (own buffer: local pointer; the others: CUDA IPC
    mappings).  torch.distributed only ships the 64-byte handles."""

    def __init__(self, comm):
        from . import ops
        self.comm, self.ops = comm, ops
        self._local, self._opened = [], []

    def alloc(self, nbytes):
        ptr, handle = self.ops.peer_alloc(int(nbytes))
        self._local.append(ptr)
        handles = [None] * self.comm.world
        dist.all_gather_object(handles, handle, group=self.comm.group)
        addrs = []
        for r, h in enumerate(handles):
            if r == self.comm.rank:
                addrs.append(ptr)
            else:
                a = self.ops.peer_open(h)
                self._opened.append(a)
                addrs.append(a)
        return addrs

    def close(self):
        torch.cuda.synchronize()
        if self.comm.world > 1:
            dist.barrier(group=self.comm.group)
        for a in self._opened:
            self.ops.peer_close(a)
        self._opened = []
        if self.comm.world > 1:
            dist.barrier(group=self.comm.group)
        for p in self._local:
            self.ops.peer_free(p)
        self._local = []


def attach_peers(engine, comm, group=None):
    """Data-parallel training without per-layer NCCL calls: gives ``engine`` the peer exchange areas that the
    single-launch BatchNorm kernels (and the loss-sum exchange) use for SyncBN over NVLink.  One slot per (layer,
    direction) plus one for the loss sums; a slot holds world x 2 x Cmax doubles."""
    if comm.world == 1:
        engine.peers = None
        return None
    group = group or PeerGroup(comm)
    cmax = max(b.cout for b in engine.dspec.blocks)
    n_slots = 2 * (len(engine.dspec.blocks) + 8) + 2
    slot_doubles = comm.world * 2 * cmax
    xchg = group.alloc(n_slots * slot_doubles * 8)
    flags = group.alloc(n_slots * 8 * 8)
    engine.comm = comm
    engine.peers = dict(world=comm.world, rank=comm.rank, xchg=xchg, flags=flags, slot_doubles=slot_doubles,
                        epoch_dev=engine.step_state.data_ptr(), n_slots=n_slots, group=group)
    return group


class ShardedTTA(object):
    """BASELINE config C4: ONE summary image, its 8 TTA transforms sharded over the ranks (unet_2d_summary.py:585-590).
    Rank 0 owns the image and the result.  Per call, inside one CUDA graph per rank:
      rank 0 publishes the image in its peer-mapped input buffer and raises every peer's `input ready` flag;
      rank r builds its transforms straight from rank 0's buffer (NVLink loads), runs the forward, and the fused head
      epilogue of dec0b stores the probabilities straight into rank 0's [8, S, S] buffer (NVLink stores), then raises its
      `probabilities ready` flag on rank 0;
      rank 0 waits for the flags and runs the fixed-order combine (bit-identical to the 1-GPU result).
    Algorithmic NVLink bytes per image: (world - 1) x (hs x ws + count x S x S) x 4."""

    def __init__(self, engine, comm, window=512, group=None):
        from . import ops
        self.eng, self.comm, self.S, self.ops = engine, comm, window, ops
        self.group = group or PeerGroup(comm)
        S = window
        self.in_addrs = self.group.alloc(S * S * 4)
        self.prob_addrs = self.group.alloc(8 * S * S * 4)
        self.flag_addrs = self.group.alloc(64 * 8)            # word 0: input ready; words 8..15: probabilities ready
        self.epoch = torch.zeros(1, dtype=torch.int64, device=engine.dev)
        self.first, self.count = shard_range(8, comm.world, comm.rank)
        self._bufs = {}

    def predict(self, summ_dev=None, hs=None, ws=None, threshold=0.5):
        """rank 0 passes the image (fp32 CUDA tensor [hs, ws]); the other ranks pass its shape.
        Returns (mask, act) device tensors on rank 0 and (None, None) elsewhere."""
        eng, ops, S, comm = self.eng, self.ops, self.S, self.comm
        if summ_dev is not None:
            hs, ws = summ_dev.shape
        key = ('sharded', hs, ws, float(threshold))
        s = eng._session(self.count, S, S, False)
        eng._ensure_inference_ready()
        st = self._bufs.get(key)
        if st is None:
            st = dict(summ=torch.zeros(hs, ws, dtype=torch.float32, device=eng.dev),
                      mask=torch.zeros(hs, ws, dtype=torch.uint8, device=eng.dev),
                      act=torch.zeros(hs, ws, dtype=torch.float64, device=eng.dev))
            self._bufs[key] = st
        if comm.rank == 0:
            st['summ'].copy_(summ_dev)
        in0 = RawTensor(self.in_addrs[0], (hs, ws), torch.float32)                     # rank 0's input buffer
        my_probs = RawTensor(self.prob_addrs[0] + self.first * S * S * 4, (self.count, S, S), torch.float32)
        all_probs = RawTensor(self.prob_addrs[0], (8, S, S), torch.float32)

        def run():
            ops.counter_advance(self.epoch)
            if comm.rank == 0:
                ops.cast_to_f32(st['summ'], in0)                                       # fp32 -> fp32 copy into the peer-visible buffer
                if comm.world > 1:
                    ops.flag_signal([self.flag_addrs[r] for r in range(1, comm.world)], self.epoch)
            else:
                ops.flag_wait(self.flag_addrs[comm.rank], 1, self.epoch)
            ops.tta_make_batch(in0, S, self.first, self.count, s['x'])
            eng._forward_inference(s, prob_out=my_probs)
            if comm.rank != 0:
                ops.flag_signal([self.flag_addrs[0] + 8 * (8 + comm.rank)], self.epoch)
            else:
                if comm.world > 1:
                    ops.flag_wait(self.flag_addrs[0] + 8 * 9, comm.world - 1, self.epoch)
                ops.tta_combine(all_probs, S, hs, ws, threshold, 8, st['act'], st['mask'])

        with torch.cuda.device(eng.dev):
            eng._run_graphed(s['tta_graphs'], key, run)
        if comm.rank != 0:
            return None, None
        return st['mask'], st['act']


def sync_parameters(engine, comm):
    """All replicas start from rank 0's weights and optimiser state."""
    for t in (engine.params, engine.nontrain, engine.adam_m, engine.adam_v, engine.step_state):
        comm.broadcast(t)
    engine._weights_dirty = True
