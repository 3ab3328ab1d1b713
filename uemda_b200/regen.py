"""Offline pseudo-label (re)generation over a whole target set, sharded over GPUs (SURVEY 8f-1, BASELINE config 4).

Reference: ``gener_target_pseudo`` (uemda/gast/pseudo_generation.py:96-155) and its refining variant
(vis_corrected_pseudo_labels.py:175-196): for every target tile
    cls  = soft class probabilities of the tile (model forward + TTA: OUTSIDE this path)
    cls  = aligner.label_refine(sup, feat, [pred1, pred2], cls, mode, temp)        (refining variant)
    cls  = pseudo_selection(cls, cutoff_top, cutoff_low, ignore_label)
    disk <- uint8(cls + 1)
The reference walks the set with batch_size=1 and round-trips every tile through ``.cpu()`` / ``torch.save``.  Here tiles
are processed in batches through the fused refine -> select chain (one C call, no host sync), the result leaves the
device as 1 byte per pixel, and the tile list is sharded over the ranks of a torch.distributed job.  File IO (PNG / .pt)
stays with the caller: ``run`` hands finished uint8 maps to a sink callback.

Exactness note: ``label_refine`` takes the *batch-global* max superpixel id as the ignored id (alignment.py:241); with
the reference's batch size of 1 that is the tile's own max.  A batch is therefore processed in one call only when all
its tiles share the same max id (always the case for maps written by the reference's edge-shrinking step, which uses
the constant H/16*W/16, superpixels.py:131,149); otherwise the batch is processed tile by tile.
"""
import torch

from . import _lib as L
from . import mining, ops

__all__ = ["PseudoLabelRegenerator"]


class PseudoLabelRegenerator:

    def __init__(self, aligner=None, cutoff_top=0.8, cutoff_low=0.6, mode="all", temp=2.0, ignore_label=-1, refine=True,
                 num_regions=None):
        self.aligner = aligner
        self.cutoff = (cutoff_top, cutoff_low, ignore_label)
        self.mode = mode
        self.temp = temp
        self.refine = refine and aligner is not None
        self.num_regions = num_regions
        self._ws = None
        self.label_hist = None   # set by run_sharded: (c+1,) int64 counts of the produced uint8 values

    # ------------------------------------------------------------------ one batch, device tensors in, uint8 out
    def _chain(self, soft, sup, feat, preds):
        views = ops.MODE_VIEWS[self.mode]
        pred1, pred2 = (preds if isinstance(preds, (list, tuple)) else (preds, None))
        out = mining.refine_select(views, soft, self.temp, feat=feat, prototypes=self.aligner.prototypes, pred1=pred1,
                                   pred2=pred2, sup=sup, num_regions=self.num_regions, eps=self.aligner.eps,
                                   select=self.cutoff, ws=self._workspace(soft, feat, pred1))
        return out[1]

    def _workspace(self, soft, feat, pred1):
        """A persistent, self-cleaning scratch buffer per batch shape when the region capacity is known; otherwise the
        chain sizes (and zero-initialises) its scratch per call."""
        if self.num_regions is None:
            return None
        b, c, H, W = soft.shape
        k = feat.shape[1] if feat is not None else 1
        low = feat if feat is not None else pred1
        h, w = (low.shape[-2], low.shape[-1]) if low is not None else (1, 1)
        key = (b, c, H, W, h, w, k, int(self.num_regions), soft.device)
        if self._ws is None or self._ws[0] != key:
            need = L.load().uem_mine_ws_bytes(b, c, H, W, h, w, k, int(self.num_regions))
            self._ws = (key, torch.zeros(int(need), dtype=torch.uint8, device=soft.device))
        return self._ws[1]

    def _count(self, u8):
        """running histogram of the produced maps over uint8 values 0 (ignored) .. c (class c-1), on the device"""
        if self.label_hist is None:
            return u8
        c = self.label_hist.numel() - 1
        # class_hist counts labels in [0, c) and, last, the non-ignored ones: feed it label - 1 with ignore = -1
        h = ops.class_hist(u8.to(torch.int64) - 1, c, -1)
        self.label_hist[1:] += h[:-1]
        self.label_hist[0] += u8.numel() - h[-1]
        return u8

    def process(self, soft, sup=None, feat=None, preds=None):
        """soft (b,c,H,W) probabilities [+ sup (b,1,H,W) int64, feat (b,k,h,w), preds] -> (b,H,W) uint8 = label + 1."""
        return self._count(self._process(soft, sup, feat, preds))

    def _process(self, soft, sup=None, feat=None, preds=None):
        L.require_cuda(soft, sup, feat)
        if not self.refine:
            from .gast.pseudo_generation import pseudo_selection
            hard = pseudo_selection(soft, self.cutoff[0], self.cutoff[1], "tensor", self.cutoff[2])
            return ops.label_plus1_u8(hard)
        views = ops.MODE_VIEWS[self.mode]
        b = soft.shape[0]
        if (views & ops.VIEW_SUP) and b > 1:
            per_tile_max = sup.reshape(b, -1).amax(dim=1)
            if not bool((per_tile_max == per_tile_max[0]).all()):  # tiles disagree on the ignored id: reference batch size 1
                parts = [self._chain(soft[i:i + 1], sup[i:i + 1], None if feat is None else feat[i:i + 1],
                                     None if preds is None else [p[i:i + 1] for p in preds] if isinstance(preds, (list, tuple))
                                     else preds[i:i + 1]) for i in range(b)]
                return ops.label_plus1_u8(torch.cat(parts))
        return ops.label_plus1_u8(self._chain(soft, sup, feat, preds))

    # ------------------------------------------------------------------ a whole (sharded) tile list
    def run(self, batches, sink, rank=0, world_size=1, device=None, store=None):
        """batches: a sequence of dicts {'soft', 'sup', 'feat', 'preds', 'names'[, 'tiles']} of HOST (ideally pinned) or
        device tensors; this rank processes the contiguous slice mining.shard_range(len(batches), rank, world_size).
        sink(names, uint8 ndarray (b,H,W)) is called once per finished batch; the array lives in one of two reused pinned
        buffers and is only valid during the call (copy what must be kept).  Input staging and the copy back are
        double-buffered.  store: a store.TileStore; every staged batch's soft labels (and superpixel maps) are then also
        written into it at the batch's 'tiles' indices, so the pass leaves the target set resident for self-training.
        Returns the number of tiles processed by this rank."""
        device = device or torch.device("cuda", torch.cuda.current_device())
        lo, hi = mining.shard_range(len(batches), rank, world_size)
        copy_stream = torch.cuda.Stream(device=device)
        cur = torch.cuda.current_stream(device)
        pending = []
        done = 0
        host_bufs = [None, None]   # pinned output buffers, reused (batch j uses buffer j % 2; at most two are in flight)

        def to_dev(x):
            if x is None:
                return None
            if isinstance(x, (list, tuple)):
                return [to_dev(y) for y in x]
            return x.to(device, non_blocking=True)

        def hand_over(x):
            # tensors staged under copy_stream are consumed by kernels on `cur`: tell the caching allocator, or their blocks
            # return to copy_stream's pool while the chain may still be reading them (the next staging would overwrite them)
            if x is None:
                return
            if isinstance(x, (list, tuple)):
                for y in x:
                    hand_over(y)
            elif x.is_cuda:
                x.record_stream(cur)

        staged = None
        for i in range(lo, hi + 1):
            nxt = None
            if i < hi:
                with torch.cuda.stream(copy_stream):  # stage batch i while batch i-1 computes
                    bt = batches[i]
                    nxt = {k: to_dev(bt.get(k)) for k in ("soft", "sup", "feat", "preds")}
                    nxt["names"] = bt.get("names")
                    nxt["tiles"] = bt.get("tiles")
                    if store is not None and nxt["tiles"] is None:
                        raise ValueError("run(store=...): every batch needs its 'tiles' indices")
                    ev = torch.cuda.Event()
                    ev.record(copy_stream)
                    nxt["ready"] = ev
            if staged is not None:
                cur.wait_event(staged["ready"])
                for k in ("soft", "sup", "feat", "preds"):
                    hand_over(staged[k])
                if store is not None:
                    store.put(staged["tiles"], staged["soft"], staged["sup"])
                u8 = self.process(staged["soft"], staged["sup"], staged["feat"], staged["preds"])
                j = (i - 1 - lo) % 2
                if host_bufs[j] is None or host_bufs[j].shape != u8.shape:
                    host_bufs[j] = torch.empty(u8.shape, dtype=torch.uint8, pin_memory=True)
                host = host_bufs[j]
                host.copy_(u8, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(cur)
                pending.append((staged["names"], host, ev, u8))
                done += u8.shape[0]
            while len(pending) > 1 or (pending and i == hi):
                names, host, ev, _keep = pending.pop(0)
                ev.synchronize()
                sink(names, host.numpy())
            staged = nxt
        return done

    # ------------------------------------------------------------------ the tile list sharded over the ranks of a job
    def run_sharded(self, batches, sink, group=None, device=None, class_num=None):
        """BASELINE config 4: the tile list sharded over the ranks of a torch.distributed job (one process per GPU,
        contiguous slices, no data-path collective).  Before the loop the prototype bank is broadcast from rank 0 and
        checked to be bit-identical everywhere (every rank refines against the same bank, as the un-sharded reference does);
        after it the class histogram of the produced label maps (uint8 values 0 = ignored, 1..c) is all-reduced, so every
        rank holds the label statistics of the WHOLE regenerated set (what ClassBalance / the IAST thresholds of the next
        self-training round start from).  Returns (tiles processed by this rank, global histogram (c+1,) int64)."""
        import torch.distributed as dist
        device = device or torch.device("cuda", torch.cuda.current_device())
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        c = class_num or (self.aligner.class_num if self.aligner is not None else None)
        assert c is not None, "class_num is needed for the label histogram"
        if world > 1 and self.aligner is not None:
            bank = self.aligner.prototypes.contiguous()
            dist.broadcast(bank, 0, group=group)
            self.aligner.prototypes = bank
            chk = torch.stack([bank.double().sum(), bank.double().abs().sum()])
            lo, hi = chk.clone(), chk.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
            assert torch.equal(lo, hi), "prototype bank differs across ranks after the broadcast"
        self.label_hist = torch.zeros(c + 1, dtype=torch.int64, device=device)
        done = self.run(batches, sink, rank=rank, world_size=world, device=device)
        hist = self.label_hist
        self.label_hist = None
        if world > 1:
            dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=group)
        return done, hist
