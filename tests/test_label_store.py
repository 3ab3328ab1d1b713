"""Resident source set (uemda_b200/store.py LabelStore, csrc/uem_store.cu label_gather_kernel): LabelStore.batch against the
torch definition (lut of the D4-cut window, then DownscaleLabel), both down-scale branches, the share / tie / ignore edges
of the cell counts, the status bits and errors, 64-bit offsets, CUDA-graph replay and the prototype update on the cut
cells.  Labels and cells are integers: every comparison is torch.equal."""
import ctypes
import re

import pytest
import torch

from oracle import uem_oracle as O
from uemda_b200.store import LabelStore

# (n_classes, byte -> label, the bytes a label file holds): ISPRS keeps its class bytes and marks 255 as ignore,
# LoveDA stores class + 1 with 0 as no-data
CONVENTIONS = {
    "isprs": (6, [-1 if v == 255 else v for v in range(256)], list(range(6)) + [255]),
    "loveda": (7, [v - 1 for v in range(256)], list(range(8))),
}


def _cut(x, y0, x0, code, Ho, Wo):
    """The window and code of uem_tile_gather: x[..., y0:y0+Hw, x0:x0+Ww] ((Hw,Ww) = (Wo,Ho) when the code transposes),
    flipped on dim -2 if bit 1, on dim -1 if bit 0, then the last two dims transposed if bit 2."""
    tr, fy, fx = (code >> 2) & 1, (code >> 1) & 1, code & 1
    Hw, Ww = (Wo, Ho) if tr else (Ho, Wo)
    x = x[..., y0:y0 + Hw, x0:x0 + Ww]
    dims = [d for d, f in ((-2, fy), (-1, fx)) if f]
    if dims:
        x = x.flip(dims)
    return x.transpose(-2, -1) if tr else x


def _ref(raw, lut, tiles, windows, Ho, Wo):
    """label[s] = lut[D4(raw[tile, window], code)]: (n,Ho,Wo) int64."""
    lut = torch.as_tensor(lut, dtype=torch.int64, device=raw.device)
    return torch.stack([lut[_cut(raw[t], y0, x0, code, Ho, Wo).long()] for t, (y0, x0, code) in zip(tiles, windows)]).contiguous()


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
            y0 = 1 + 2 * int(torch.randint(0, (my + 1) // 2, (1,), generator=g))
            x0 = 1 + 2 * int(torch.randint(0, (mx + 1) // 2, (1,), generator=g))
        else:
            y0 = int(torch.randint(0, my + 1, (1,), generator=g))
            x0 = int(torch.randint(0, mx + 1, (1,), generator=g))
        out.append((y0, x0, code))
    return out


def _label_bytes(T, H, W, valid, g, block=24, noise=0.1):
    """Blocky label maps (block x block patches of one byte, a share `noise` of pixels redrawn) so that cells have
    majorities above and below min_ratio; every byte from `valid`."""
    valid = torch.tensor(valid, dtype=torch.uint8)
    low = torch.randint(0, len(valid), (T, -(-H // block), -(-W // block)), generator=g)
    idx = low.repeat_interleave(block, 1).repeat_interleave(block, 2)[:, :H, :W]
    flip = torch.rand(T, H, W, generator=g) < noise
    idx = torch.where(flip, torch.randint(0, len(valid), (T, H, W), generator=g), idx)
    return valid[idx]


# ------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("code", range(8))
def test_cells_are_window_blocks(code):
    """The definition on the CPU (oracle DownscaleLabel): output cell (cy, cx) of a cut label is the majority of one
    s x s block of the window, whatever the order of its pixels.  The floor drops the trailing output rows and columns,
    which lie at the start of the window under a flip (the kernel counts a cell's pixels wherever they lie in the tile)."""
    g = torch.Generator().manual_seed(code)
    C, lut, valid = CONVENTIONS["loveda"]
    s, Ho, Wo = 4, 18, 13                       # 4 x 3 cells; 2 rows and 1 column dropped
    raw = _label_bytes(1, 40, 40, valid, g, block=3, noise=0.3)
    y0, x0 = 5, 7
    label = _ref(raw, lut, [0], [(y0, x0, code)], Ho, Wo)
    down = O.downscale_label(label, s, C, -1, 0.75)
    assert down.shape == (1, 1, Ho // s, Wo // s)
    tr, fy, fx = (code >> 2) & 1, (code >> 1) & 1, code & 1
    win = torch.as_tensor(lut)[_cut(raw[0], y0, x0, 0, *((Wo, Ho) if tr else (Ho, Wo))).long()]
    for cy in range(Ho // s):
        for cx in range(Wo // s):
            # output rows [cy*s, cy*s+s) are window rows (columns if transposed), counted from the end under a flip
            rows, cols = (cx, cy) if tr else (cy, cx)
            flip_r, flip_c = (fy, fx)
            Hw, Ww = win.shape
            r0 = Hw - (rows + 1) * s if flip_r else rows * s
            c0 = Ww - (cols + 1) * s if flip_c else cols * s
            block = win[r0:r0 + s, c0:c0 + s].reshape(-1)
            shuffled = block[torch.randperm(block.numel(), generator=g)].reshape(1, s, s)
            assert int(down[0, 0, cy, cx]) == int(O.downscale_label(shuffled, s, C, -1, 0.75)[0, 0, 0, 0]), (cy, cx)


def test_lut_is_validated_at_construction():
    with pytest.raises(ValueError):
        LabelStore(2, 8, 8, list(range(255)), device="cpu")
    with pytest.raises(ValueError):
        LabelStore(2, 8, 8, torch.zeros(2, 128, dtype=torch.int64), device="cpu")
    with pytest.raises(TypeError):
        LabelStore(2, 8, 8, torch.zeros(256), device="cpu")


def test_store_refuses_a_cpu_device():
    from uemda_b200._lib import UemLibraryError
    with pytest.raises(UemLibraryError):
        LabelStore(2, 8, 8, list(range(256)), device="cpu")


@pytest.fixture(scope="module")
def lib():
    from uemda_b200 import _lib, build
    build.build()
    return _lib.load()


def test_bad_arguments_are_refused(lib):
    """Refused before any pointer is touched (so this runs without a device)."""
    p = ctypes.c_void_p(256)   # never dereferenced

    def call(label, scale, n_classes, down):
        return lib.uem_label_gather_u8(p, 4, 64, 64, p, p, p, 2, 32, 32, label, scale, n_classes, -1, 0.75, down, p, None)

    for label, scale, n_classes, down, what in ((None, 16, 6, None, b"no output"),
                                                (p, 16, 9, p, b"n_classes"), (p, 16, 0, p, b"n_classes"),
                                                (p, 1, 6, p, b"scale"), (p, 0, 6, p, b"scale"), (p, -16, 6, p, b"scale"),
                                                (None, 12, 6, p, b"label_out"), (None, 32, 6, p, b"label_out")):
        assert call(label, scale, n_classes, down) != 0, (label, scale, n_classes, down)
        assert what in lib.uem_last_error(), lib.uem_last_error()
    assert lib.uem_label_gather_u8(p, 4, 64, 64, None, p, p, 2, 32, 32, p, 0, 0, -1, 0.75, None, p, None) != 0   # no lut
    assert lib.uem_label_gather_u8(p, 4, 64, 64, p, p, p, 65536, 32, 32, p, 0, 0, -1, 0.75, None, p, None) != 0


# ------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from uemda_b200 import _lib
    _lib.load()
    return torch.device("cuda", 0)


def _filled(T, Hs, Ws, conv, dev, seed):
    """A store of blocky label bytes, filled through put from pinned host memory; returns the store and the host bytes."""
    C, lut, valid = CONVENTIONS[conv]
    raw = _label_bytes(T, Hs, Ws, valid, torch.Generator().manual_seed(seed)).pin_memory()
    st = LabelStore(T, Hs, Ws, lut, device=dev)
    st.put(list(range(T)), raw.unsqueeze(1))
    return st, raw


def _check(st, C, tiles, windows, Ho, Wo, scale):
    from uemda_b200 import ops
    from uemda_b200.gast.alignment import DownscaleLabel
    ds = DownscaleLabel(scale, C, -1, 0.75)
    label, down = st.batch(tiles, windows, (Ho, Wo), downscale=ds)
    want = _ref(st.raw, st.lut, tiles, windows, Ho, Wo)
    assert label.dtype == torch.int64 and label.shape == (len(tiles), Ho, Wo)
    assert torch.equal(label, want), (windows, Ho, Wo)
    assert down.shape == (len(tiles), 1, Ho // scale, Wo // scale)
    assert torch.equal(down, ops.downscale_label(want, scale, C, -1, 0.75)), (windows, Ho, Wo, scale)
    alone, none = st.batch(tiles, windows, (Ho, Wo))
    assert none is None and torch.equal(alone, want)


@pytest.mark.gpu
@pytest.mark.parametrize("tile", [(512, 512), (1024, 1024), (97, 130)])
@pytest.mark.parametrize("scale", [16, 8, 4, 2, 12, 32])
def test_gather_matches_torch(dev, tile, scale):
    """16 / 8 / 4 / 2: counted in the gather's launch; 12 / 32: the gather, then uem_downscale_label_i64.  Square and
    non-square tiles and windows, 512^2 crops of 1024^2 tiles, Ho / Wo not multiples of the scale under every code."""
    Hs, Ws = tile
    T = 5
    g = torch.Generator().manual_seed(Hs * 100 + scale)
    for conv in CONVENTIONS:
        C = CONVENTIONS[conv][0]
        st, raw = _filled(T, Hs, Ws, conv, dev, seed=Hs + scale)
        assert torch.equal(st.raw.cpu(), raw)
        m = min(Hs, Ws)
        calls = [(list(range(4)), Hs, Ws, "full"), (list(range(4, 8)), Ws, Hs, "full")]
        if Hs == 1024:
            calls += [(list(range(8)), 512, 512, "any")]                  # the LoveDA training crop
        calls += [(list(range(8)), m // 2, m // 2, "odd"),
                  (list(range(8)), m - 5, m - 3, "edge"),
                  (list(range(8)), m // 2 + 3, m // 3 + 1, "any")]
        for codes, Ho, Wo, place in calls:
            cs = codes * (16 // len(codes))
            tiles = torch.randint(0, T, (len(cs),), generator=g).tolist()
            tiles[1] = tiles[0]
            _check(st, C, tiles, _windows(cs, Hs, Ws, Ho, Wo, place, g), Ho, Wo, scale)
            _check(st, C, [T - 1], _windows(codes[-1:], Hs, Ws, Ho, Wo, place, g), Ho, Wo, scale)
        del st
        torch.cuda.empty_cache()


def _edge_tile(s, C, ignore_byte, byte_of, g):
    """One s-row tile of 6 cells with known counts (pixels shuffled within each cell), and the cells' expected labels at
    min_ratio 0.75 and 0.5.  byte_of(class) is the stored byte of a class."""
    a = s * s
    keep = -(-3 * a // 4)            # exactly 3/4 (192 of 256 at s = 16)
    cells = [  # (counts as {byte: count}, expected at 0.75, expected at 0.5)
        ({byte_of(2): keep, byte_of(1): a - keep}, 2, 2),
        ({byte_of(2): keep - 1, byte_of(1): a - keep + 1}, -1, 2),                   # one pixel short of 3/4
        ({ignore_byte: keep, byte_of(0): a - keep}, -1, -1),                         # ignore majority
        ({byte_of(C - 1): a // 2, byte_of(3): a // 2}, -1, 3),                       # tie: the lower class index
        ({ignore_byte: a // 2, byte_of(C - 1): a // 2}, -1, C - 1),                  # class tied with ignore: the class
        ({byte_of(C - 1): a}, C - 1, C - 1),
    ]
    tile = torch.empty(s, 6 * s, dtype=torch.uint8)
    for i, (counts, _, _) in enumerate(cells):
        px = torch.cat([torch.full((cnt,), b, dtype=torch.uint8) for b, cnt in counts.items()])
        tile[:, i * s:(i + 1) * s] = px[torch.randperm(a, generator=g)].view(s, s)
    return tile, [c[1] for c in cells], [c[2] for c in cells]


@pytest.mark.gpu
@pytest.mark.parametrize("conv", ["isprs", "loveda"])
@pytest.mark.parametrize("scale", [16, 8, 4])
def test_downscale_edges_fused(dev, conv, scale):
    from uemda_b200 import ops
    from uemda_b200.gast.alignment import DownscaleLabel
    C, lut, valid = CONVENTIONS[conv]
    ignore_byte = 255 if conv == "isprs" else 0
    g = torch.Generator().manual_seed(scale)
    tile, want75, want50 = _edge_tile(scale, C, ignore_byte, (lambda c: c) if conv == "isprs" else (lambda c: c + 1), g)
    st = LabelStore(1, scale, 6 * scale, lut, device=dev)
    st.put([0], tile[None].to(dev))
    for ratio, want in ((0.75, want75), (0.5, want50)):
        ds = DownscaleLabel(scale, C, -1, ratio)
        label, down = st.batch([0], [(0, 0, 0)], (scale, 6 * scale), downscale=ds)
        assert down.view(-1).tolist() == want, (ratio, down.view(-1).tolist())
        for code in range(8):   # every code permutes the cells' pixels: same cells, in the code's order
            Ho, Wo = (6 * scale, scale) if code & 4 else (scale, 6 * scale)
            label, down = st.batch([0], [(0, 0, code)], (Ho, Wo), downscale=ds)
            assert torch.equal(down, ops.downscale_label(_ref(st.raw, lut, [0], [(0, 0, code)], Ho, Wo), scale, C, -1, ratio))
            assert sorted(down.view(-1).tolist()) == sorted(want)
    assert int(st.status.item()) == 0


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name.replace(" ", "") for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return {nm for nm in names if not nm.lower().startswith(("memcpy", "memset"))}


@pytest.mark.gpu
def test_each_branch_launches_its_kernels(dev):
    """Power-of-two scales <= 16: the gather kernel alone.  12 and 32: the gather kernel, then the generic / pow2
    DownscaleLabel kernel.  No downscale: the gather kernel alone."""
    from uemda_b200.gast.alignment import DownscaleLabel
    C, lut, _ = CONVENTIONS["loveda"]
    st, _ = _filled(2, 128, 128, "loveda", dev, seed=1)
    tiles = torch.tensor([0, 1], dtype=torch.int64, device=dev)
    wins = torch.tensor([(0, 0, 0), (3, 5, 6)], dtype=torch.int32, device=dev)
    gather = r"(?<![A-Za-z0-9_])label_gather_kernel"
    for scale, other in ((16, None), (8, None), (4, None), (2, None), (12, r"downscale_kernel<7>"),
                         (32, r"downscale_pow2_kernel<7>"), (None, None)):
        ds = DownscaleLabel(scale, C, -1, 0.75) if scale else None
        names = _kernel_names(lambda: st.batch(tiles, wins, (96, 96), downscale=ds))
        assert any(re.search(gather, nm) for nm in names), (scale, sorted(names))
        if other is None:
            assert len(names) == 1, (scale, sorted(names))
        else:
            assert len(names) == 2 and any(re.search(r"(?<![A-Za-z0-9_])" + other, nm) for nm in names), (scale, sorted(names))


@pytest.mark.gpu
def test_cells_without_labels(dev):
    """label_out = NULL: a power-of-two scale <= 16 writes the cells alone, equal to those of a call with labels."""
    from uemda_b200 import _lib as L
    C, lut, _ = CONVENTIONS["isprs"]
    st, _ = _filled(3, 200, 160, "isprs", dev, seed=4)
    g = torch.Generator().manual_seed(4)
    tiles = torch.tensor([2, 0, 1, 1], dtype=torch.int64, device=dev)
    wins = torch.tensor(_windows([0, 3, 5, 6], 200, 160, 90, 70, "any", g), dtype=torch.int32, device=dev)
    for scale in (16, 8, 4, 2):
        down = torch.full((4, 1, 90 // scale, 70 // scale), 99, dtype=torch.int64, device=dev)
        L.check(L.bind(st.raw).uem_label_gather_u8(L.ptr(st.raw), 3, 200, 160, L.ptr(st.lut), L.ptr(tiles), L.ptr(wins), 4, 90, 70,
                                                   None, scale, C, -1, 0.75, L.ptr(down), L.ptr(st.status), L.stream_of(st.raw)))
        from uemda_b200.gast.alignment import DownscaleLabel
        _, want = st.batch(tiles, wins, (90, 70), downscale=DownscaleLabel(scale, C, -1, 0.75))
        assert torch.equal(down, want), scale


@pytest.mark.gpu
def test_out_of_range_samples(dev, monkeypatch):
    from uemda_b200 import config
    from uemda_b200.gast.alignment import DownscaleLabel
    C, lut, _ = CONVENTIONS["loveda"]
    T, Hs, Ws, Ho, Wo = 4, 64, 80, 32, 48
    st, _ = _filled(T, Hs, Ws, "loveda", dev, seed=3)
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
    for scale in (16, 12):
        out = (torch.full((n, Ho, Wo), 7, dtype=torch.int64, device=dev),
               torch.full((n, 1, Ho // scale, Wo // scale), 7, dtype=torch.int64, device=dev))
        label, down = st.batch(dt, dw, (Ho, Wo), downscale=DownscaleLabel(scale, C, -1, 0.75), out=out)
        torch.cuda.synchronize()
        assert int(st.status.item()) == 1
        want = _ref(st.raw, lut, tiles[:3], good, Ho, Wo)
        assert torch.equal(label[:3], want)
        from uemda_b200 import ops
        assert torch.equal(down[:3], ops.downscale_label(want, scale, C, -1, 0.75))
        assert not label[3:].any() and not down[3:].any()
        st.status.zero_()
    # a clean batch leaves the status alone; under strict_asserts a bad sample raises and the word is cleared
    st.batch(tiles[:3], good, (Ho, Wo))
    assert int(st.status.item()) == 0
    monkeypatch.setattr(config, "strict_asserts", True)
    st.batch(tiles[:3], good, (Ho, Wo), downscale=DownscaleLabel(16, C, -1, 0.75))
    with pytest.raises(IndexError):
        st.batch([T], [(0, 0, 0)], (Ho, Wo))
    assert int(st.status.item()) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [16, 12])
def test_labels_outside_the_classes(dev, monkeypatch, scale):
    """A LUT value outside {ignore} U [0, n_classes) sets bit 1 and raises DownscaleLabel's error, only with downscale.
    The check covers every label of the window, the trailing rows that no cell holds included (the reference's one_hot
    takes the whole label map).  Such labels are not counted, as in uem_downscale_label_i64."""
    from uemda_b200 import config, ops
    from uemda_b200.gast.alignment import DownscaleLabel
    C, _, _ = CONVENTIONS["isprs"]
    lut = [-1 if v == 255 else v for v in range(256)]   # bytes 6..254 are outside the 6 classes
    T, Hs, Ws, Ho, Wo = 2, 64, 64, 40, 48
    raw = torch.zeros(T, Hs, Ws, dtype=torch.uint8)
    raw[0, :24, :24] = 3
    raw[0, 5, 5] = 9                                 # inside a cell
    raw[1, Ho - 1, 2] = 200                          # in the last row: no cell of scale 16 or 12 holds it
    st = LabelStore(T, Hs, Ws, lut, device=dev)
    st.put([0, 1], raw)
    ds = DownscaleLabel(scale, C, -1, 0.75)
    monkeypatch.setattr(config, "strict_asserts", False)
    for t in (0, 1):
        label, down = st.batch([t], [(0, 0, 0)], (Ho, Wo))        # without downscale: the labels as mapped, no error
        assert int(st.status.item()) == 0 and torch.equal(label, _ref(st.raw, lut, [t], [(0, 0, 0)], Ho, Wo))
        assert int(label.max()) == (9 if t == 0 else 200)
        label, down = st.batch([t], [(0, 0, 0)], (Ho, Wo), downscale=ds)
        assert int(st.status.item()) == 2, t
        assert torch.equal(down, ops.downscale_label(label, scale, C, -1, 0.75))
        st.status.zero_()
    monkeypatch.setattr(config, "strict_asserts", True)
    st.batch([1], [(0, 0, 0)], (Ho, Wo))
    for t in (0, 1):
        with pytest.raises(RuntimeError, match="Class values must be non-negative and smaller than num_classes."):
            st.batch([t], [(0, 0, 0)], (Ho, Wo), downscale=ds)
        assert int(st.status.item()) == 0


@pytest.mark.gpu
def test_bad_arguments_are_refused_gpu(dev):
    from uemda_b200._lib import UemLibraryError
    from uemda_b200.gast.alignment import DownscaleLabel
    _, lut, _ = CONVENTIONS["isprs"]
    st = LabelStore(2, 32, 32, lut, device=dev)
    with pytest.raises(UemLibraryError, match="n_classes"):
        st.batch([0], [(0, 0, 0)], 32, downscale=DownscaleLabel(16, 9, -1, 0.75))
    with pytest.raises(ValueError):
        LabelStore(2, 32, 32, lut[:255], device=dev)
    with pytest.raises(TypeError):
        st.put([0], torch.zeros(1, 32, 32, dtype=torch.int64, device=dev))
    with pytest.raises(IndexError):
        st.put([2], torch.zeros(1, 32, 32, dtype=torch.uint8, device=dev))
    with pytest.raises(ValueError):
        st.batch([0], [(0, 0, 0)], 32, downscale=DownscaleLabel(16, 6, -1, 0.75),
                 out=(torch.empty(1, 32, 32, dtype=torch.int64, device=dev), None))


@pytest.mark.gpu
def test_store_past_2g_bytes(dev):
    """8200 tiles of 512^2 = 2.15e9 bytes: the last tiles lie past byte 2^31."""
    from uemda_b200 import ops
    from uemda_b200.gast.alignment import DownscaleLabel
    C, lut, valid = CONVENTIONS["loveda"]
    T, H, W = 8200, 512, 512
    assert (T - 1) * H * W > 2 ** 31
    st = LabelStore(T, H, W, lut, device=dev)
    g = torch.Generator().manual_seed(7)
    last = list(range(T - 4, T))
    raw = _label_bytes(4, H, W, valid, g)
    st.put(last, raw.to(dev))
    codes = list(range(8))
    tiles = [last[i % 4] for i in codes]
    wins = _windows(codes, H, W, 300, 200, "any", g)
    label, down = st.batch(tiles, wins, (300, 200), downscale=DownscaleLabel(16, C, -1, 0.75))
    want = _ref(raw, lut, [t - (T - 4) for t in tiles], wins, 300, 200).to(dev)
    assert torch.equal(label, want)
    assert torch.equal(down, ops.downscale_label(want, 16, C, -1, 0.75))
    assert torch.equal(st.raw[T - 1].cpu(), raw[3])
    del st, label, down, want
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [16, 12])
def test_cuda_graph_replay(dev, monkeypatch, scale):
    from uemda_b200 import config
    from uemda_b200.gast.alignment import DownscaleLabel
    monkeypatch.setattr(config, "strict_asserts", False)
    C, lut, _ = CONVENTIONS["loveda"]
    T, Hs, Ws, Ho, Wo, n = 6, 256, 256, 128, 128, 8
    st, _ = _filled(T, Hs, Ws, "loveda", dev, seed=11)
    ds = DownscaleLabel(scale, C, -1, 0.75)
    g = torch.Generator().manual_seed(5)

    def draw():
        codes = torch.randint(0, 8, (n,), generator=g).tolist()
        return torch.randint(0, T, (n,), generator=g).tolist(), _windows(codes, Hs, Ws, Ho, Wo, "any", g)

    t0, w0 = draw()
    dt = torch.tensor(t0, dtype=torch.int64, device=dev)
    dw = torch.tensor(w0, dtype=torch.int32, device=dev)
    out = (torch.empty(n, Ho, Wo, dtype=torch.int64, device=dev),
           torch.empty(n, 1, Ho // scale, Wo // scale, dtype=torch.int64, device=dev))
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        st.batch(dt, dw, (Ho, Wo), downscale=ds, out=out)   # warm-up outside the capture
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        st.batch(dt, dw, (Ho, Wo), downscale=ds, out=out)
    for _ in range(3):
        tl, wl = draw()
        dt.copy_(torch.tensor(tl, dtype=torch.int64))
        dw.copy_(torch.tensor(wl, dtype=torch.int32))
        graph.replay()
        label, down = st.batch(tl, wl, (Ho, Wo), downscale=ds)
        torch.cuda.synchronize()
        assert torch.equal(out[0], label) and torch.equal(out[1], down)
        assert torch.equal(out[0], _ref(st.raw, lut, tl, wl, Ho, Wo))
    assert int(st.status.item()) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("conv", ["isprs", "loveda"])
def test_prototype_update_on_the_cut_cells(dev, conv):
    """cfg2 shape (8 x 512^2 out of 512^2 tiles, all 8 codes): _compute_local_prototypes on the cells of batch(...) gives
    the bank of update_prototype on the labels, bit for bit (the reference's alignment.py:86-90 with the downscale done)."""
    from uemda_b200.gast.alignment import Aligner

    class _Log:
        def info(self, *a, **k):
            pass

    C, lut, _ = CONVENTIONS[conv]
    st, _ = _filled(8, 512, 512, conv, dev, seed=21)
    g = torch.Generator().manual_seed(21)
    feat = torch.randn(8, 64, 32, 32, generator=g).to(dev)
    bank = torch.randn(C, 64, generator=g).to(dev)
    tiles = [3, 1, 4, 1, 5, 0, 2, 6]
    wins = [(0, 0, code) for code in range(8)]
    a1, a2 = Aligner(_Log(), feat_channels=64, class_num=C, decay=0.996), Aligner(_Log(), feat_channels=64, class_num=C, decay=0.996)
    a1.prototypes, a2.prototypes = bank.clone(), bank.clone()
    label, down = st.batch(tiles, wins, 512, downscale=a2.downscale_gt)
    a2._compute_local_prototypes(feat, down, update=True, decay=a2.decay)
    want_down = a1.update_prototype(feat, label)
    assert torch.equal(down, want_down)
    assert (down >= 0).any() and (down < 0).any()
    assert torch.equal(a1.prototypes, a2.prototypes)
    assert not torch.equal(a1.prototypes, bank)
