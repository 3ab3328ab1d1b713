"""Resident image set (uemda_b200/store.py ImageStore, csrc/uem_store.cu image_gather_kernel): ImageStore.batch against the
torch definition (each channel's table of the D4-cut window), both store forms, the alignment of the cut pixels with those
of TileStore and LabelStore, the status bit and errors, 64-bit offsets and CUDA-graph replay; normalize_table against a
numpy restatement of albumentations' Normalize.  The cut is a permutation and the lookup exact: every comparison is exact."""
import ctypes
import re

import numpy as np
import pytest
import torch

from uemda_b200.store import ImageStore, LabelStore, TileStore

IMAGENET = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))


def _cut(x, y0, x0, code, Ho, Wo):
    """The window and code of uem_tile_gather on (..., H, W): x[..., y0:y0+Hw, x0:x0+Ww] ((Hw,Ww) = (Wo,Ho) when the code
    transposes), flipped on dim -2 if bit 1, on dim -1 if bit 0, then the last two dims transposed if bit 2."""
    tr, fy, fx = (code >> 2) & 1, (code >> 1) & 1, code & 1
    Hw, Ww = (Wo, Ho) if tr else (Ho, Wo)
    x = x[..., y0:y0 + Hw, x0:x0 + Ww]
    dims = [d for d, f in ((-2, fy), (-1, fx)) if f]
    if dims:
        x = x.flip(dims)
    return x.transpose(-2, -1) if tr else x


def _ref(raw, table, tiles, windows, Ho, Wo):
    """image[s, ch] = table[ch][D4(raw[tile, window, ch])]: (n,C,Ho,Wo) fp32 from a (T,H,W,C) uint8 store."""
    table = table.to(raw.device)
    ch = torch.arange(table.shape[0], device=raw.device).view(-1, 1, 1)
    return torch.stack([table[ch, _cut(raw[t].permute(2, 0, 1), y0, x0, code, Ho, Wo).long()]
                        for t, (y0, x0, code) in zip(tiles, windows)]).contiguous()


def _windows(codes, Hs, Ws, Ho, Wo, place, g):
    """Per code, a window (y0, x0) that fits the tile: 'full' at the origin, 'odd' at odd offsets, 'edge' touching the
    right and bottom edges, 'any' anywhere."""
    out = []
    for code in codes:
        Hw, Ww = (Wo, Ho) if code & 4 else (Ho, Wo)
        my, mx = Hs - Hw, Ws - Ww
        assert my >= 0 and mx >= 0
        if place == "full":
            y0 = x0 = 0
        elif place == "edge":
            y0, x0 = my, mx
        elif place == "odd":
            assert my >= 1 and mx >= 1
            y0 = 1 + 2 * int(torch.randint(0, (my + 1) // 2, (1,), generator=g))
            x0 = 1 + 2 * int(torch.randint(0, (mx + 1) // 2, (1,), generator=g))
        else:
            y0 = int(torch.randint(0, my + 1, (1,), generator=g))
            x0 = int(torch.randint(0, mx + 1, (1,), generator=g))
        out.append((y0, x0, code))
    return out


def _albumentations_normalize(img, mean, std, max_pixel_value=255.0):
    """albumentations.augmentations.functional.normalize, restated: float32 in-place arithmetic on an HWC image."""
    mean = np.array(mean, dtype=np.float32)
    mean *= max_pixel_value
    std = np.array(std, dtype=np.float32)
    std *= max_pixel_value
    denominator = np.reciprocal(std, dtype=np.float32)
    img = img.astype(np.float32)
    img -= mean
    img *= denominator
    return img


# ------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("mean,std,max_pixel_value", [
    (IMAGENET[0], IMAGENET[1], 255.0),                                             # statistics on the [0, 1] scale
    (tuple(255 * m for m in IMAGENET[0]), tuple(255 * s for s in IMAGENET[1]), 1.0),   # the same on the byte scale
    ((0.5, 0.5, 0.5, 0.5), (0.5, 0.5, 0.5, 0.5), 255.0),
    ((0.0,), (1.0,), 1.0),
])
def test_normalize_table_is_albumentations_normalize(mean, std, max_pixel_value):
    table = ImageStore.normalize_table(mean, std, max_pixel_value)
    C = len(mean)
    assert table.dtype == torch.float32 and table.shape == (C, 256)
    img = np.repeat(np.arange(256, dtype=np.uint8)[:, None], C, axis=1)[None]       # (1, 256, C): every byte in every channel
    want = _albumentations_normalize(img, mean, std, max_pixel_value)[0].T            # (C, 256)
    assert np.array_equal(table.numpy().view(np.int32), np.ascontiguousarray(want).view(np.int32))


def test_table_and_channels_are_validated_at_construction():
    table = ImageStore.normalize_table(*IMAGENET)
    for channels in (0, 5):
        with pytest.raises(ValueError):
            ImageStore(2, 8, 8, channels, torch.zeros(max(channels, 1), 256), device="cpu")
    with pytest.raises(ValueError):
        ImageStore(2, 8, 8, 3, table[:2], device="cpu")
    with pytest.raises(ValueError):
        ImageStore(2, 8, 8, 3, table.t(), device="cpu")
    with pytest.raises(ValueError):
        ImageStore(2, 8, 8, 3, table.reshape(-1), device="cpu")
    with pytest.raises(ValueError):
        ImageStore(2, 8, 8, 3, table[:, :255], device="cpu")
    with pytest.raises(TypeError):
        ImageStore(2, 8, 8, 3, torch.zeros(3, 256, dtype=torch.int64), device="cpu")
    with pytest.raises(TypeError):
        ImageStore(2, 8, 8, 3, torch.zeros(3, 256, dtype=torch.uint8), device="cpu")


def test_store_refuses_a_cpu_device():
    from uemda_b200._lib import UemLibraryError
    with pytest.raises(UemLibraryError):
        ImageStore(2, 8, 8, 3, ImageStore.normalize_table(*IMAGENET), device="cpu")


@pytest.fixture(scope="module")
def lib():
    from uemda_b200 import _lib, build
    build.build()
    return _lib.load()


def test_bad_arguments_are_refused(lib):
    """Refused before any pointer is touched (so this runs without a device)."""
    p = ctypes.c_void_p(256)   # never dereferenced

    def call(C=3, table=p, out=p, n=2, Ho=32):
        return lib.uem_image_gather_u8(p, 4, 64, 64, C, table, p, p, n, Ho, 32, out, p, None)

    for kw, what in (({"C": 0}, b"channels"), ({"C": 5}, b"channels"), ({"C": -1}, b"channels"),
                     ({"table": None}, b"bad arguments"), ({"out": None}, b"bad arguments"),
                     ({"n": 65536}, b"bad arguments"), ({"n": -1}, b"bad arguments"), ({"Ho": 0}, b"bad arguments"),
                     ({"Ho": 16 * 65536}, b"too large")):
        assert call(**kw) != 0, kw
        assert what in lib.uem_last_error(), (kw, lib.uem_last_error())


# ------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from uemda_b200 import _lib
    _lib.load()
    return torch.device("cuda", 0)


def _table(C, g):
    """Distinct random values per channel, so that a byte read from the wrong channel maps to the wrong value."""
    return torch.randn(C, 256, generator=g)


def _filled(T, Hs, Ws, C, dev, seed):
    """A store of random image bytes, filled through put from pinned host memory; returns the store and the host bytes."""
    g = torch.Generator().manual_seed(seed)
    raw = torch.randint(0, 256, (T, Hs, Ws, C), generator=g, dtype=torch.uint8).pin_memory()
    st = ImageStore(T, Hs, Ws, C, _table(C, g), device=dev)
    st.put(list(range(T)), raw)
    return st, raw


def _check(st, tiles, windows, Ho, Wo):
    img = st.batch(tiles, windows, (Ho, Wo))
    assert img.dtype == torch.float32 and img.shape == (len(tiles), st.shape[3], Ho, Wo)
    assert torch.equal(img, _ref(st.raw, st.table, tiles, windows, Ho, Wo)), (windows, Ho, Wo)


@pytest.mark.gpu
@pytest.mark.parametrize("tile", [(512, 512), (1024, 1024), (97, 130)])
@pytest.mark.parametrize("C", [1, 3, 4])
def test_gather_matches_torch(dev, tile, C):
    """All 8 codes on square and non-square tiles and windows, 512^2 crops of 1024^2 tiles, at the origin, at odd offsets,
    at the edge and anywhere; Ho / Wo include sizes that are not multiples of 16, 64 or 4 (the 4-byte store form)."""
    Hs, Ws = tile
    T = 5
    g = torch.Generator().manual_seed(Hs * 10 + C)
    st, raw = _filled(T, Hs, Ws, C, dev, seed=Hs + C)
    assert torch.equal(st.raw.cpu(), raw)
    m = min(Hs, Ws)
    calls = [(list(range(4)), Hs, Ws, "full"), (list(range(4, 8)), Ws, Hs, "full")]
    if Hs == 1024:
        calls += [(list(range(8)), 512, 512, "any")]                  # the LoveDA training crop
    calls += [(list(range(8)), m // 2, m // 2, "odd"),
              (list(range(8)), m - 5, m - 3, "edge"),
              (list(range(8)), m // 2 + 3, m // 3 + 1, "any"),
              (list(range(8)), m // 2 + 1, m // 2 + 4, "any")]      # Wo % 4 == 0 with an odd Ho
    for codes, Ho, Wo, place in calls:
        cs = codes * (16 // len(codes))
        tiles = torch.randint(0, T, (len(cs),), generator=g).tolist()
        tiles[1] = tiles[0]
        _check(st, tiles, _windows(cs, Hs, Ws, Ho, Wo, place, g), Ho, Wo)
        _check(st, [T - 1], _windows(codes[-1:], Hs, Ws, Ho, Wo, place, g), Ho, Wo)


@pytest.mark.gpu
def test_flips_keep_the_channel_order(dev):
    """Every pixel holds the bytes (1, 2, 3): under every code each plane is constant.  A kernel that reverses the bytes of
    a row under a horizontal flip, instead of its pixels, swaps channels 0 and 2."""
    st = ImageStore(1, 40, 70, 3, torch.arange(256, dtype=torch.float32).expand(3, 256), device=dev)
    st.put([0], torch.tensor([1, 2, 3], dtype=torch.uint8, device=dev).expand(1, 40, 70, 3).contiguous())
    for code in range(8):
        Ho, Wo = (33, 21) if code & 4 else (21, 33)
        img = st.batch([0], [(3, 5, code)], (Ho, Wo))
        for ch in range(3):
            assert bool((img[0, ch] == ch + 1).all()), code


def _offset(t, elems):
    """Contiguous zero tensor of t's shape whose data pointer sits `elems` elements past a 256-byte boundary."""
    buf = torch.zeros(t.numel() + 64 + elems, dtype=t.dtype, device=t.device)
    start = (-buf.data_ptr() % 256) // t.element_size() + elems
    v = buf[start:start + t.numel()].view(t.shape)
    assert v.is_contiguous() and v.data_ptr() % 256 == elems * t.element_size()
    return v


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name.replace(" ", "") for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return {nm for nm in names if not nm.lower().startswith(("memcpy", "memset"))}


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 2, 3, 4])
def test_each_store_form_is_launched(dev, C):
    """16-byte stores (<C,4>) when Wo % 4 == 0 and out is 16-byte aligned; 4-byte stores (<C,1>) when Wo % 4 != 0 or out
    is not 16-byte aligned.  Each launch alone, each equal to the torch definition."""
    T, Hs, Ws = 3, 160, 200
    st, _ = _filled(T, Hs, Ws, C, dev, seed=30 + C)
    g = torch.Generator().manual_seed(C)
    for Ho, Wo, off, form in ((96, 128, 0, 4), (61, 76, 0, 4), (96, 126, 0, 1), (61, 77, 0, 1), (96, 128, 1, 1),
                              (96, 128, 2, 1), (61, 76, 3, 1)):
        codes = list(range(8))
        tiles = torch.randint(0, T, (8,), generator=g).to(dev)
        wins = torch.tensor(_windows(codes, Hs, Ws, Ho, Wo, "any", g), dtype=torch.int32, device=dev)
        out = _offset(torch.empty(8, C, Ho, Wo, device=dev), off)
        names = _kernel_names(lambda: st.batch(tiles, wins, (Ho, Wo), out=out))
        pat = re.compile(r"(?<![A-Za-z0-9_])image_gather_kernel<%d,%d>" % (C, form))
        assert len(names) == 1 and pat.search(next(iter(names))), (Ho, Wo, off, sorted(names))
        assert torch.equal(out, _ref(st.raw, st.table, tiles.tolist(), wins.tolist(), Ho, Wo)), (Ho, Wo, off)


def _coded_tiles(T, H, W):
    """Tile t's pixel (y, x) has the id t*H*W + y*W + x; the image holds its 4 little-endian bytes."""
    ids = (torch.arange(T, dtype=torch.int64).view(T, 1, 1) * H * W + torch.arange(H * W, dtype=torch.int64).view(1, H, W))
    img = torch.stack([(ids >> (8 * k)) & 255 for k in range(4)], -1).to(torch.uint8)
    return ids, img


@pytest.mark.gpu
@pytest.mark.parametrize("tile,size", [((96, 128), (40, 72)), ((1024, 1024), (512, 512))])
def test_same_pixels_as_the_label_stores(dev, tile, size):
    """One (tiles, windows) set cut from an ImageStore, a TileStore and a LabelStore of the same tiles: under every code,
    every pixel of the image names the same tile pixel as the superpixel id and the label byte of that pixel."""
    T, (H, W), (Ho, Wo) = 3, tile, size
    ids, img = _coded_tiles(T, H, W)
    im = ImageStore(T, H, W, 4, torch.arange(256, dtype=torch.float32).expand(4, 256), device=dev)
    im.put(list(range(T)), img.to(dev))
    ts = TileStore(T, 1, H, W, device=dev)
    ts.put(list(range(T)), torch.zeros(T, 1, H, W, device=dev), ids.to(torch.int32).to(dev))
    ls = LabelStore(T, H, W, list(range(256)), device=dev)
    ls.put(list(range(T)), (ids % 251).to(torch.uint8).to(dev))
    g = torch.Generator().manual_seed(H)
    codes = list(range(8)) * 2
    tiles = torch.randint(0, T, (16,), generator=g).tolist()
    wins = _windows(codes, H, W, Ho, Wo, "any", g)
    got = im.batch(tiles, wins, (Ho, Wo)).to(torch.int64)
    got = got[:, 0] | got[:, 1] << 8 | got[:, 2] << 16 | got[:, 3] << 24                   # (n,Ho,Wo) ids
    _, sup = ts.batch(tiles, wins, (Ho, Wo))
    label, _ = ls.batch(tiles, wins, (Ho, Wo))
    assert torch.equal(got, sup[:, 0])
    assert torch.equal(got % 251, label)
    assert torch.equal(got // (H * W), torch.tensor(tiles, device=dev).view(-1, 1, 1).expand_as(got))


@pytest.mark.gpu
def test_out_of_range_samples(dev, monkeypatch):
    from uemda_b200 import config
    T, Hs, Ws, Ho, Wo, C = 4, 64, 80, 32, 48, 3
    st, _ = _filled(T, Hs, Ws, C, dev, seed=3)
    good = [(0, 0, 0), (5, 7, 6), (Hs - Ho, Ws - Wo, 3)]
    bad_tiles = [(-1, (0, 0, 0)), (T, (0, 0, 0)), (2 ** 40, (0, 0, 5))]
    bad_windows = [(1, (Hs - Ho + 1, 0, 0)), (1, (0, Ws - Wo + 1, 1)), (1, (-1, 0, 2)), (1, (0, -2, 0)),
                   (1, (Hs - Wo + 1, 0, 4)), (1, (0, Ws - Ho + 1, 7)), (1, (0, 0, 8)), (1, (0, 0, -1))]
    tiles = [2, 1, 3] + [t for t, _ in bad_tiles + bad_windows]
    wins = good + [w for _, w in bad_tiles + bad_windows]
    n = len(tiles)
    dt = torch.tensor(tiles, dtype=torch.int64, device=dev)
    dw = torch.tensor(wins, dtype=torch.int32, device=dev)
    monkeypatch.setattr(config, "strict_asserts", False)
    for off in (0, 1):   # both store forms
        out = _offset(torch.empty(n, C, Ho, Wo, device=dev), off).fill_(7.0)
        img = st.batch(dt, dw, (Ho, Wo), out=out)
        torch.cuda.synchronize()
        assert img is out and int(st.status.item()) == 1
        assert torch.equal(img[:3], _ref(st.raw, st.table, tiles[:3], good, Ho, Wo))
        assert not img[3:].any()
        st.status.zero_()
    # a clean batch leaves the status alone; under strict_asserts a bad sample raises and the word is cleared
    st.batch(tiles[:3], good, (Ho, Wo))
    assert int(st.status.item()) == 0
    monkeypatch.setattr(config, "strict_asserts", True)
    st.batch(tiles[:3], good, (Ho, Wo))
    for t, w in bad_tiles[:1] + bad_windows[:1]:
        with pytest.raises(IndexError):
            st.batch([t], [w], (Ho, Wo))
        assert int(st.status.item()) == 0


@pytest.mark.gpu
def test_bad_arguments_are_refused_gpu(dev):
    st = ImageStore(2, 32, 32, 3, ImageStore.normalize_table(*IMAGENET), device=dev)
    for bad in (torch.zeros(1, 32, 32, 3, dtype=torch.int64, device=dev), torch.zeros(1, 32, 32, 3, device=dev)):
        with pytest.raises(TypeError):
            st.put([0], bad)
    for bad in (torch.zeros(1, 32, 32, dtype=torch.uint8, device=dev), torch.zeros(1, 3, 32, 32, dtype=torch.uint8, device=dev),
                torch.zeros(1, 32, 32, 4, dtype=torch.uint8, device=dev), torch.zeros(1, 32, 31, 3, dtype=torch.uint8, device=dev)):
        with pytest.raises(ValueError):
            st.put([0], bad)
    with pytest.raises(IndexError):
        st.put([2], torch.zeros(1, 32, 32, 3, dtype=torch.uint8, device=dev))
    with pytest.raises(ValueError):
        st.put([0, 1], torch.zeros(1, 32, 32, 3, dtype=torch.uint8, device=dev))
    with pytest.raises(ValueError):
        st.batch(torch.tensor([0, 1], device=dev), torch.zeros(1, 3, dtype=torch.int32, device=dev), 16)
    for bad in (torch.empty(1, 3, 16, 16, dtype=torch.float64, device=dev), torch.empty(1, 3, 16, 17, device=dev),
                torch.empty(2, 3, 16, 16, device=dev), torch.empty(1, 16, 16, 3, device=dev).permute(0, 3, 1, 2),
                torch.empty(1, 3, 16, 16), (torch.empty(1, 3, 16, 16, device=dev),)):
        with pytest.raises(ValueError):
            st.batch([0], [(0, 0, 0)], 16, out=bad)
    assert int(st.status.item()) == 0


@pytest.mark.gpu
def test_store_past_2g_bytes(dev):
    """2800 tiles of 512^2 x 3 = 2.2e9 bytes: the last tiles lie past byte 2^31."""
    T, H, W, C = 2800, 512, 512, 3
    assert (T - 1) * H * W * C > 2 ** 31
    g = torch.Generator().manual_seed(7)
    st = ImageStore(T, H, W, C, _table(C, g), device=dev)
    last = list(range(T - 4, T))
    raw = torch.randint(0, 256, (4, H, W, C), generator=g, dtype=torch.uint8)
    st.put(last, raw.to(dev))
    codes = list(range(8))
    tiles = [last[i % 4] for i in codes]
    wins = _windows(codes, H, W, 300, 200, "any", g)
    img = st.batch(tiles, wins, (300, 200))
    assert torch.equal(img, _ref(raw.to(dev), st.table, [t - (T - 4) for t in tiles], wins, 300, 200))
    assert torch.equal(st.raw[T - 1].cpu(), raw[3])
    del st, img
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("Wo", [128, 127])
def test_cuda_graph_replay(dev, monkeypatch, Wo):
    from uemda_b200 import config
    monkeypatch.setattr(config, "strict_asserts", False)
    T, Hs, Ws, Ho, n, C = 6, 256, 256, 128, 8, 3
    st, _ = _filled(T, Hs, Ws, C, dev, seed=11)
    g = torch.Generator().manual_seed(5)

    def draw():
        codes = torch.randint(0, 8, (n,), generator=g).tolist()
        return torch.randint(0, T, (n,), generator=g).tolist(), _windows(codes, Hs, Ws, Ho, Wo, "any", g)

    t0, w0 = draw()
    dt = torch.tensor(t0, dtype=torch.int64, device=dev)
    dw = torch.tensor(w0, dtype=torch.int32, device=dev)
    out = torch.empty(n, C, Ho, Wo, device=dev)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        st.batch(dt, dw, (Ho, Wo), out=out)   # warm-up outside the capture
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        st.batch(dt, dw, (Ho, Wo), out=out)
    for _ in range(3):
        tl, wl = draw()
        dt.copy_(torch.tensor(tl, dtype=torch.int64))
        dw.copy_(torch.tensor(wl, dtype=torch.int32))
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, _ref(st.raw, st.table, tl, wl, Ho, Wo))
    assert int(st.status.item()) == 0


@pytest.mark.gpu
def test_normalized_batch_is_the_normalized_crop(dev):
    """The intended use: a store with normalize_table gives, per sample, albumentations' normalize of the host-side crop /
    flip / rot90 (TileStore.d4_code) of the decoded image, bit for bit."""
    T, H, W, C = 3, 200, 180, 3
    g = torch.Generator().manual_seed(2)
    raw = torch.randint(0, 256, (T, H, W, C), generator=g, dtype=torch.uint8)
    st = ImageStore(T, H, W, C, ImageStore.normalize_table(*IMAGENET), device=dev)
    st.put(list(range(T)), raw.pin_memory())
    idx, win, want = [], [], []
    for k in range(4):
        for hflip in (False, True):
            for vflip in (False, True):
                t = len(idx) % T
                y0, x0 = 3 * k + 1, 5 * k + (2 if hflip else 0)
                crop = raw[t, y0:y0 + 96, x0:x0 + 96]                                    # HWC
                if hflip:
                    crop = crop.flip(1)
                if vflip:
                    crop = crop.flip(0)
                crop = torch.rot90(crop, k, dims=(0, 1))
                want.append(torch.from_numpy(_albumentations_normalize(crop.numpy(), *IMAGENET)).permute(2, 0, 1))
                idx.append(t)
                win.append((y0, x0, TileStore.d4_code(rot90=k, hflip=hflip, vflip=vflip)))
    got = st.batch(idx, win, 96)
    assert torch.equal(got.cpu(), torch.stack(want))
