"""Resident target set (SURVEY 8f-1): the target tiles' soft labels and superpixel maps kept in HBM, each training batch
cut from them on the device.

Reference: ``gener_target_pseudo`` writes every tile's soft probabilities with ``torch.save`` (pseudo_generation.py:135-136);
during self-training the loader reads them back with the int32 superpixel .tif (basedata.py:77-79,87), applies the same
crop / flip / rot90 to both (augmentation.py:150-157) and the step copies them to the device (train_ssl_uem.py:199-201).
Here the loader returns ``(index, y0, x0, code)`` per sample and ``TileStore.batch`` produces ``label_t_soft`` (n,c,Ho,Wo)
fp32 and ``label_t_sup`` (n,1,Ho,Wo) int64 in one launch (uem_tile_gather): only the augmentation parameters cross PCIe.
"""
import torch

from . import _lib as L
from . import config

__all__ = ["TileStore"]

_I32_MIN, _I32_MAX = -2 ** 31, 2 ** 31 - 1


class TileStore:
    """``soft``: (T,c,H,W) fp32 and ``ids``: (T,H,W) int32 (the reference's on-disk type, superpixels.py:113,150), each one
    allocation, zero until ``put``.  ``superpixels=False`` keeps soft labels only (``ids`` is None)."""

    def __init__(self, num_tiles, class_num, height, width, device=None, superpixels=True):
        device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if device.type != "cuda":
            raise L.UemLibraryError("TileStore lives on a CUDA device (got %s)" % device)
        self.shape = (int(num_tiles), int(class_num), int(height), int(width))
        self.soft = torch.zeros(self.shape, dtype=torch.float32, device=device)
        self.ids = torch.zeros((self.shape[0],) + self.shape[2:], dtype=torch.int32, device=device) if superpixels else None
        # bit 0: a sample of a batch() named a tile outside the store or a window outside the tile
        self.status = torch.zeros(1, dtype=torch.int32, device=device)

    @property
    def device(self):
        return self.soft.device

    @staticmethod
    def d4_code(rot90=0, hflip=False, vflip=False):
        """The gather code of the augmentation "hflip (dim -1), then vflip (dim -2), then torch.rot90(x, rot90, dims=(-2, -1))".
        The code means: flip dim -2 if bit 1, flip dim -1 if bit 0, then transpose the last two dims if bit 2.  torch.rot90
        by 1 is flip(-1) then transpose, by 2 is flip(-2, -1), by 3 is flip(-2) then transpose."""
        k = int(rot90) % 4
        fx, fy = int(bool(hflip)), int(bool(vflip))
        if k in (1, 2):
            fx ^= 1
        if k in (2, 3):
            fy ^= 1
        return ((k & 1) << 2) | (fy << 1) | fx

    def _tile_list(self, tiles, b):
        tiles = [int(t) for t in (tiles.tolist() if torch.is_tensor(tiles) else tiles)]
        if len(tiles) != b:
            raise ValueError("put: %d tile indices for a batch of %d" % (len(tiles), b))
        bad = [t for t in tiles if not 0 <= t < self.shape[0]]
        if bad:
            raise IndexError("put: tile index %d outside [0, %d)" % (bad[0], self.shape[0]))
        return tiles

    def put(self, tiles, soft, sup=None):
        """Writes soft (b,c,H,W) and, if given, sup ((b,1,H,W) or (b,H,W), int64 or int32) at the tile indices ``tiles``
        (a sequence or a tensor of b indices).  Inputs may be on the host (pinned: the copies are asynchronous) or on the
        device; copies run on the current stream.  Under config.strict_asserts ids outside the int32 range raise (one
        read-back); otherwise they are truncated like the int64 -> int32 cast."""
        b = soft.shape[0]
        if tuple(soft.shape[1:]) != self.shape[1:]:
            raise ValueError("put: soft labels of shape %s do not fit a store of %s" % (tuple(soft.shape), self.shape))
        if sup is not None:
            if self.ids is None:
                raise ValueError("put: this store was made without superpixels")
            if sup.dim() == 4:
                if sup.shape[1] != 1:
                    raise ValueError("put: superpixel maps must be (b,1,H,W) or (b,H,W)")
                sup = sup[:, 0]
            if tuple(sup.shape) != (b,) + self.shape[2:]:
                raise ValueError("put: superpixel maps of shape %s do not fit a store of %s" % (tuple(sup.shape), self.shape))
            if sup.dtype not in (torch.int64, torch.int32):
                raise TypeError("put: superpixel ids must be int64 or int32 (got %s)" % sup.dtype)
            if config.strict_asserts and sup.dtype == torch.int64 and sup.numel():
                lo, hi = int(sup.min()), int(sup.max())
                if lo < _I32_MIN or hi > _I32_MAX:
                    raise RuntimeError("put: superpixel id %d outside the int32 range of the store" % (lo if lo < _I32_MIN else hi))
        tiles = self._tile_list(tiles, b)
        # one copy per run of consecutive tile indices
        i = 0
        while i < b:
            j = i + 1
            while j < b and tiles[j] == tiles[j - 1] + 1:
                j += 1
            t = tiles[i]
            self.soft[t:t + j - i].copy_(soft[i:j], non_blocking=True)
            if sup is not None:
                self.ids[t:t + j - i].copy_(sup[i:j], non_blocking=True)
            i = j

    def _stage(self, tiles, windows):
        """Host index lists -> device tensors with one small copy; device tensors pass through (graph-capturable)."""
        dev = self.device
        if torch.is_tensor(tiles) and tiles.is_cuda and torch.is_tensor(windows) and windows.is_cuda:
            return (tiles.to(device=dev, dtype=torch.int64).contiguous().view(-1),
                    windows.to(device=dev, dtype=torch.int32).contiguous().view(-1, 3))
        t = torch.as_tensor(tiles.cpu() if torch.is_tensor(tiles) else tiles, dtype=torch.int64).reshape(-1)
        w = torch.as_tensor(windows.cpu() if torch.is_tensor(windows) else windows, dtype=torch.int32).reshape(-1, 3)
        n = t.numel()
        host = torch.empty(5 * n, dtype=torch.int32, pin_memory=True)   # [n int64 tiles | n x 3 int32 windows]
        host[:2 * n].view(torch.int64).copy_(t)
        host[2 * n:].copy_(w.reshape(-1))
        staged = host.to(dev, non_blocking=True)
        return staged[:2 * n].view(torch.int64), staged[2 * n:].view(-1, 3)

    def batch(self, tiles, windows, size, out=None):
        """Cuts one batch: sample s is ``store[tiles[s]]`` at window (y0, x0) = windows[s][:2] under code windows[s][2]
        (``d4_code``), size = (Ho, Wo) or an int.  Returns (soft (n,c,Ho,Wo) fp32, sup (n,1,Ho,Wo) int64, or None without
        superpixels), written into ``out`` = (soft, sup) when given.  tiles (n,) int64 / windows (n,3) int32 device tensors
        and ``out`` make the call capturable in a CUDA graph (with config.strict_asserts off); host sequences are staged
        with one small copy.  Under config.strict_asserts an out-of-range sample raises (one read-back of the status word,
        which is then cleared); otherwise its outputs are zero and ``status`` keeps bit 0 set."""
        Ho, Wo = (int(size), int(size)) if isinstance(size, int) else (int(size[0]), int(size[1]))
        tiles, windows = self._stage(tiles, windows)
        n = tiles.numel()
        if windows.shape[0] != n:
            raise ValueError("batch: %d tile indices but %d windows" % (n, windows.shape[0]))
        T, c, H, W = self.shape
        if out is None:
            soft = torch.empty((n, c, Ho, Wo), dtype=torch.float32, device=self.device)
            sup = None if self.ids is None else torch.empty((n, 1, Ho, Wo), dtype=torch.int64, device=self.device)
        else:
            soft, sup = out
            if (soft.shape != (n, c, Ho, Wo) or soft.dtype != torch.float32 or soft.device != self.device
                    or not soft.is_contiguous()):
                raise ValueError("batch: out soft must be a contiguous (%d,%d,%d,%d) fp32 tensor on %s" % (n, c, Ho, Wo, self.device))
            if self.ids is not None and (sup is None or sup.shape != (n, 1, Ho, Wo) or sup.dtype != torch.int64
                                         or sup.device != self.device or not sup.is_contiguous()):
                raise ValueError("batch: out sup must be a contiguous (%d,1,%d,%d) int64 tensor on %s" % (n, Ho, Wo, self.device))
            if self.ids is None:
                sup = None
        lib = L.bind(self.soft)
        L.check(lib.uem_tile_gather(L.ptr(self.soft), L.ptr(self.ids), T, c, H, W, L.ptr(tiles), L.ptr(windows), n, Ho, Wo,
                                    L.ptr(soft), L.ptr(sup), L.ptr(self.status), L.stream_of(self.soft)))
        if config.strict_asserts:
            bits = int(self.status.item())
            if bits:
                self.status.zero_()
                raise IndexError("TileStore.batch: a sample names a tile outside [0, %d) or a window outside the %dx%d tile"
                                 % (T, H, W))
        return soft, sup
