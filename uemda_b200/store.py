"""Resident target set (SURVEY 8f-1): the target tiles' soft labels and superpixel maps kept in HBM, each training batch
cut from them on the device.

Reference: ``gener_target_pseudo`` writes every tile's soft probabilities with ``torch.save`` (pseudo_generation.py:135-136);
during self-training the loader reads them back with the int32 superpixel .tif (basedata.py:77-79,87), applies the same
crop / flip / rot90 to both (augmentation.py:150-157) and the step copies them to the device (train_ssl_uem.py:199-201).
Here the loader returns ``(index, y0, x0, code)`` per sample and ``TileStore.batch`` produces ``label_t_soft`` (n,c,Ho,Wo)
fp32 and ``label_t_sup`` (n,1,Ho,Wo) int64 in one launch (uem_tile_gather): only the augmentation parameters cross PCIe.

Resident source set: the source label files' bytes kept in HBM.  The loader decodes the label PNG, crops / flips / rotates it,
widens it to int64 (train_ssl_uem.py:205,216, train_align_uem.py:147,150) and the step down-scales it again for the
prototypes (alignment.py:86-90,484-509).  ``LabelStore.batch`` produces ``label_s`` and its DownscaleLabel cells in one
launch (uem_label_gather_u8) from the same ``(index, y0, x0, code)`` per sample.

Resident image set: the decoded images' bytes kept in HBM.  The loader crops / flips / rotates each image with its labels
(augmentation.py:150-157), normalises it to fp32 and the step copies the batch to the device.  ``ImageStore.batch`` cuts the
normalised batch in one launch (uem_image_gather_u8) from the same ``(index, y0, x0, code)``, so the host only draws them.
"""
import numpy as np
import torch

from . import _lib as L
from . import config
from .ops import f32

__all__ = ["TileStore", "LabelStore", "ImageStore"]

_I32_MIN, _I32_MAX = -2 ** 31, 2 ** 31 - 1


def _cuda_device(device, what):
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if device.type != "cuda":
        raise L.UemLibraryError("%s lives on a CUDA device (got %s)" % (what, device))
    return device


def _tile_list(tiles, b, num_tiles):
    tiles = [int(t) for t in (tiles.tolist() if torch.is_tensor(tiles) else tiles)]
    if len(tiles) != b:
        raise ValueError("put: %d tile indices for a batch of %d" % (len(tiles), b))
    bad = [t for t in tiles if not 0 <= t < num_tiles]
    if bad:
        raise IndexError("put: tile index %d outside [0, %d)" % (bad[0], num_tiles))
    return tiles


def _runs(tiles):
    """(first tile, i, j) per run tiles[i:j] of consecutive tile indices: one copy each."""
    i, b = 0, len(tiles)
    while i < b:
        j = i + 1
        while j < b and tiles[j] == tiles[j - 1] + 1:
            j += 1
        yield tiles[i], i, j
        i = j


def _stage(tiles, windows, dev):
    """Host index lists -> device tensors with one small copy; device tensors pass through (graph-capturable)."""
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


def _size(size):
    return (int(size), int(size)) if isinstance(size, int) else (int(size[0]), int(size[1]))


class TileStore:
    """``soft``: (T,c,H,W) fp32 and ``ids``: (T,H,W) int32 (the reference's on-disk type, superpixels.py:113,150), each one
    allocation, zero until ``put``.  ``superpixels=False`` keeps soft labels only (``ids`` is None)."""

    def __init__(self, num_tiles, class_num, height, width, device=None, superpixels=True):
        device = _cuda_device(device, "TileStore")
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
        for t, i, j in _runs(_tile_list(tiles, b, self.shape[0])):
            self.soft[t:t + j - i].copy_(soft[i:j], non_blocking=True)
            if sup is not None:
                self.ids[t:t + j - i].copy_(sup[i:j], non_blocking=True)

    def batch(self, tiles, windows, size, out=None):
        """Cuts one batch: sample s is ``store[tiles[s]]`` at window (y0, x0) = windows[s][:2] under code windows[s][2]
        (``d4_code``), size = (Ho, Wo) or an int.  Returns (soft (n,c,Ho,Wo) fp32, sup (n,1,Ho,Wo) int64, or None without
        superpixels), written into ``out`` = (soft, sup) when given.  tiles (n,) int64 / windows (n,3) int32 device tensors
        and ``out`` make the call capturable in a CUDA graph (with config.strict_asserts off); host sequences are staged
        with one small copy.  Under config.strict_asserts an out-of-range sample raises (one read-back of the status word,
        which is then cleared); otherwise its outputs are zero and ``status`` keeps bit 0 set."""
        Ho, Wo = _size(size)
        tiles, windows = _stage(tiles, windows, self.device)
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


class LabelStore:
    """``raw``: (T,H,W) uint8, the source label files' own bytes, one allocation, zero until ``put``.  ``lut``: 256 int64
    on the device, the loader's byte -> label mapping (LoveDA: ``0 -> -1, v -> v - 1``; an ignore byte: ``255 -> -1``),
    validated here.  ``batch`` cuts a batch with the windows and codes of ``TileStore.batch`` (``TileStore.d4_code``)."""

    def __init__(self, num_tiles, height, width, lut, device=None):
        lut = torch.as_tensor(lut)
        if lut.dim() != 1 or lut.numel() != 256:
            raise ValueError("LabelStore: lut must map each of the 256 byte values (got shape %s)" % (tuple(lut.shape),))
        if lut.is_floating_point() or lut.is_complex() or lut.dtype == torch.bool:
            raise TypeError("LabelStore: lut must hold integer labels (got %s)" % lut.dtype)
        device = _cuda_device(device, "LabelStore")
        self.shape = (int(num_tiles), int(height), int(width))
        self.raw = torch.zeros(self.shape, dtype=torch.uint8, device=device)
        self.lut = lut.to(device=device, dtype=torch.int64).contiguous()
        # bit 0: a sample of a batch() named a tile outside the store or a window outside the tile;
        # bit 1: a batch() with downscale met a label outside {ignore} U [0, n_classes)
        self.status = torch.zeros(1, dtype=torch.int32, device=device)

    @property
    def device(self):
        return self.raw.device

    def put(self, tiles, raw):
        """Writes raw (b,H,W) or (b,1,H,W) uint8 label bytes at the tile indices ``tiles`` (a sequence or a tensor of b
        indices), from the host (pinned: the copies are asynchronous) or the device, on the current stream."""
        if raw.dtype != torch.uint8:
            raise TypeError("put: label bytes must be uint8 (got %s)" % raw.dtype)
        if raw.dim() == 4:
            if raw.shape[1] != 1:
                raise ValueError("put: label maps must be (b,1,H,W) or (b,H,W)")
            raw = raw[:, 0]
        if raw.dim() != 3 or tuple(raw.shape[1:]) != self.shape[1:]:
            raise ValueError("put: label maps of shape %s do not fit a store of %s" % (tuple(raw.shape), self.shape))
        for t, i, j in _runs(_tile_list(tiles, raw.shape[0], self.shape[0])):
            self.raw[t:t + j - i].copy_(raw[i:j], non_blocking=True)

    def batch(self, tiles, windows, size, downscale=None, out=None):
        """Cuts one batch: label[s] = lut[store[tiles[s]] at window (y0, x0) = windows[s][:2] under code windows[s][2]],
        size = (Ho, Wo) or an int, and with ``downscale`` (a DownscaleLabel, e.g. ``aligner.downscale_gt``) its cells
        down[s] = downscale(label[s]) in the same launch.  Returns (label (n,Ho,Wo) int64, down (n,1,Ho//s,Wo//s) int64 or
        None), written into ``out`` = (label, down) when given.  tiles (n,) int64 / windows (n,3) int32 device tensors and
        ``out`` make the call capturable in a CUDA graph (with config.strict_asserts off).  An out-of-range sample gets a
        zero label (and the cells of a zero map) and sets bit 0 of ``status``; with ``downscale``, a label outside
        {ignore} U [0, n_classes) sets bit 1 and is not counted.  Under config.strict_asserts the call reads the word back,
        clears it and raises IndexError for bit 0, or DownscaleLabel's RuntimeError for bit 1."""
        Ho, Wo = _size(size)
        tiles, windows = _stage(tiles, windows, self.device)
        n = tiles.numel()
        if windows.shape[0] != n:
            raise ValueError("batch: %d tile indices but %d windows" % (n, windows.shape[0]))
        T, H, W = self.shape
        scale = n_classes = ignore = 0
        min_ratio = 0.0
        if downscale is not None:
            scale, n_classes = int(downscale.scale_factor), int(downscale.n_classes)
            ignore, min_ratio = int(downscale.ignore_label), f32(downscale.min_ratio)
        dshape = (n, 1, Ho // scale, Wo // scale) if downscale is not None else None
        if out is None:
            label = torch.empty((n, Ho, Wo), dtype=torch.int64, device=self.device)
            down = torch.empty(dshape, dtype=torch.int64, device=self.device) if dshape else None
        else:
            label, down = out
            for name, t, shape in (("label", label, (n, Ho, Wo)), ("down", down, dshape)):
                if shape and (t is None or t.shape != shape or t.dtype != torch.int64 or t.device != self.device
                              or not t.is_contiguous()):
                    raise ValueError("batch: out %s must be a contiguous %s int64 tensor on %s" % (name, shape, self.device))
            if dshape is None:
                down = None
        lib = L.bind(self.raw)
        L.check(lib.uem_label_gather_u8(L.ptr(self.raw), T, H, W, L.ptr(self.lut), L.ptr(tiles), L.ptr(windows), n, Ho, Wo,
                                        L.ptr(label), scale, n_classes, ignore, min_ratio, L.ptr(down), L.ptr(self.status),
                                        L.stream_of(self.raw)))
        if config.strict_asserts:
            bits = int(self.status.item())
            if bits:
                self.status.zero_()
                if bits & 1:
                    raise IndexError("LabelStore.batch: a sample names a tile outside [0, %d) or a window outside the %dx%d "
                                     "tile" % (T, H, W))
                # F.one_hot in the reference (alignment.py:502) rejects these
                raise RuntimeError("Class values must be non-negative and smaller than num_classes.")
        return label, down


class ImageStore:
    """``raw``: (T,H,W,C) uint8, the decoded images' bytes as image files hold them (channels interleaved, C in [1,4]: RGB,
    IRRG, RGB+IR), one allocation, zero until ``put``.  ``table``: (C,256) fp32 on the device, the byte -> value map of each
    channel (``normalize_table`` for albumentations' Normalize; ``torch.arange(256.) / 255`` per channel for ToTensor),
    validated here.  ``batch`` cuts a batch with the windows and codes of ``TileStore.batch`` (``TileStore.d4_code``), so the
    same indices and windows cut the same pixels out of a ``TileStore`` / ``LabelStore`` of the same tiles."""

    def __init__(self, num_tiles, height, width, channels, table, device=None):
        channels = int(channels)
        if not 1 <= channels <= 4:
            raise ValueError("ImageStore: %d channels outside [1, 4]" % channels)
        table = torch.as_tensor(table)
        if tuple(table.shape) != (channels, 256):
            raise ValueError("ImageStore: table must map each of the 256 byte values of each of the %d channels, shape (%d, 256) "
                             "(got %s)" % (channels, channels, tuple(table.shape)))
        if not table.is_floating_point():
            raise TypeError("ImageStore: table must hold floating-point values (got %s)" % table.dtype)
        device = _cuda_device(device, "ImageStore")
        self.shape = (int(num_tiles), int(height), int(width), channels)
        self.raw = torch.zeros(self.shape, dtype=torch.uint8, device=device)
        self.table = table.to(device=device, dtype=torch.float32).contiguous()
        # bit 0: a sample of a batch() named a tile outside the store or a window outside the tile
        self.status = torch.zeros(1, dtype=torch.int32, device=device)

    @property
    def device(self):
        return self.raw.device

    @staticmethod
    def normalize_table(mean, std, max_pixel_value=255.0):
        """(C,256) fp32 table of albumentations' ``Normalize(mean, std, max_pixel_value)`` with its arithmetic, in float32:
        ``(v - mean * max_pixel_value) * reciprocal(std * max_pixel_value)``."""
        m = np.asarray(mean, dtype=np.float32) * np.float32(max_pixel_value)
        s = np.asarray(std, dtype=np.float32) * np.float32(max_pixel_value)
        r = np.reciprocal(s, dtype=np.float32)
        v = np.arange(256, dtype=np.float32)
        return torch.from_numpy(np.ascontiguousarray((v[None, :] - m[:, None]) * r[:, None], dtype=np.float32))

    def put(self, tiles, images):
        """Writes images (b,H,W,C) uint8 at the tile indices ``tiles`` (a sequence or a tensor of b indices), from the host
        (pinned: the copies are asynchronous) or the device, on the current stream."""
        if images.dtype != torch.uint8:
            raise TypeError("put: image bytes must be uint8 (got %s)" % images.dtype)
        if images.dim() != 4 or tuple(images.shape[1:]) != self.shape[1:]:
            raise ValueError("put: images of shape %s do not fit a store of %s (b,H,W,C)" % (tuple(images.shape), self.shape))
        for t, i, j in _runs(_tile_list(tiles, images.shape[0], self.shape[0])):
            self.raw[t:t + j - i].copy_(images[i:j], non_blocking=True)

    def batch(self, tiles, windows, size, out=None):
        """Cuts one batch: image[s, ch] = table[ch][store[tiles[s], ..., ch] at window (y0, x0) = windows[s][:2] under code
        windows[s][2]], size = (Ho, Wo) or an int.  Returns (n,C,Ho,Wo) fp32, written into ``out`` when given.  tiles (n,)
        int64 / windows (n,3) int32 device tensors and ``out`` make the call capturable in a CUDA graph (with
        config.strict_asserts off).  An out-of-range sample gets zero planes and sets bit 0 of ``status``; under
        config.strict_asserts the call reads the word back, clears it and raises IndexError."""
        Ho, Wo = _size(size)
        tiles, windows = _stage(tiles, windows, self.device)
        n = tiles.numel()
        if windows.shape[0] != n:
            raise ValueError("batch: %d tile indices but %d windows" % (n, windows.shape[0]))
        T, H, W, C = self.shape
        if out is None:
            out = torch.empty((n, C, Ho, Wo), dtype=torch.float32, device=self.device)
        elif (not torch.is_tensor(out) or out.shape != (n, C, Ho, Wo) or out.dtype != torch.float32 or out.device != self.device
              or not out.is_contiguous()):
            raise ValueError("batch: out must be a contiguous (%d,%d,%d,%d) fp32 tensor on %s" % (n, C, Ho, Wo, self.device))
        lib = L.bind(self.raw)
        L.check(lib.uem_image_gather_u8(L.ptr(self.raw), T, H, W, C, L.ptr(self.table), L.ptr(tiles), L.ptr(windows), n, Ho, Wo,
                                        L.ptr(out), L.ptr(self.status), L.stream_of(self.raw)))
        if config.strict_asserts:
            if int(self.status.item()):
                self.status.zero_()
                raise IndexError("ImageStore.batch: a sample names a tile outside [0, %d) or a window outside the %dx%d tile"
                                 % (T, H, W))
        return out
