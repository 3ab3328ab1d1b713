"""Resident target set (uemda_b200/store.py, csrc/uem_store.cu): TileStore.batch against the torch expression that defines
the gather code, the D4 code of an augmentation, out-of-range samples, 64-bit offsets, CUDA-graph replay, the regeneration
hook and the mining chain on a gathered batch.  The gather is a permutation copy: every comparison is torch.equal."""
import pytest
import torch

from uemda_b200.store import TileStore


def _ref(soft, ids, tiles, windows, Ho, Wo):
    """The definition of uem_tile_gather: window store[tile, :, y0:y0+Hw, x0:x0+Ww] ((Hw,Ww) = (Wo,Ho) when the code
    transposes), flipped on dim -2 if bit 1, on dim -1 if bit 0, then the last two dims transposed if bit 2."""
    outs_s, outs_i = [], []
    for t, (y0, x0, code) in zip(tiles, windows):
        tr, fy, fx = (code >> 2) & 1, (code >> 1) & 1, code & 1
        Hw, Ww = (Wo, Ho) if tr else (Ho, Wo)

        def cut(x):
            x = x[..., y0:y0 + Hw, x0:x0 + Ww]
            dims = [d for d, f in ((-2, fy), (-1, fx)) if f]
            if dims:
                x = x.flip(dims)
            return x.transpose(-2, -1) if tr else x

        outs_s.append(cut(soft[t]))
        if ids is not None:
            outs_i.append(cut(ids[t]).to(torch.int64).unsqueeze(0))
    return torch.stack(outs_s).contiguous(), (torch.stack(outs_i).contiguous() if ids is not None else None)


def _augment(x, rot90, hflip, vflip):
    if hflip:
        x = x.flip(-1)
    if vflip:
        x = x.flip(-2)
    return torch.rot90(x, rot90, dims=(-2, -1))


# ------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("rot90", [0, 1, 2, 3])
@pytest.mark.parametrize("hflip", [False, True])
@pytest.mark.parametrize("vflip", [False, True])
def test_d4_code_matches_flip_rot90(rot90, hflip, vflip):
    x = torch.arange(2 * 5 * 7, dtype=torch.float32).view(1, 2, 5, 7)   # one non-square tile, c = 2
    want = _augment(x[0], rot90, hflip, vflip)
    code = TileStore.d4_code(rot90, hflip, vflip)
    got, _ = _ref(x, None, [0], [(0, 0, code)], want.shape[-2], want.shape[-1])
    assert torch.equal(got[0], want)


def test_d4_codes_are_the_eight_group_elements():
    codes = {TileStore.d4_code(r, h, v) for r in range(4) for h in (False, True) for v in (False, True)}
    assert codes == set(range(8))
    assert TileStore.d4_code(-1) == TileStore.d4_code(3) and TileStore.d4_code(5, True) == TileStore.d4_code(1, True)


def test_transposing_codes_take_a_transposed_window():
    x = torch.arange(1 * 1 * 9 * 11, dtype=torch.float32).view(1, 1, 9, 11)
    for code in range(8):
        got, _ = _ref(x, None, [0], [(1, 2, code)], 4, 6)
        assert got.shape == (1, 1, 4, 6)
        # the window of a transposing code is 6 rows x 4 columns: its first output row is a window column
        first_row = x[0, 0, 1:7, 2:6] if code & 4 else x[0, 0, 1:5, 2:8]
        assert sorted(got[0, 0].flatten().tolist()) == sorted(first_row.flatten().tolist())


def test_store_refuses_a_cpu_device():
    from uemda_b200._lib import UemLibraryError
    with pytest.raises(UemLibraryError):
        TileStore(2, 6, 8, 8, device="cpu")


# ------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from uemda_b200 import _lib
    _lib.load()
    return torch.device("cuda", 0)


def _filled(T, c, Hs, Ws, dev, seed, superpixels=True):
    """A store with random soft labels and ids (including both ends of the int32 range), filled through put from pinned
    host memory; returns the store and the host copies."""
    g = torch.Generator().manual_seed(seed)
    soft = torch.rand(T, c, Hs, Ws, generator=g).pin_memory()
    ids = None
    if superpixels:
        ids = torch.randint(-3, 5000, (T, 1, Hs, Ws), generator=g, dtype=torch.int64)
        ids.view(-1)[:2] = torch.tensor([2 ** 31 - 1, -2 ** 31])
        ids = ids.pin_memory()
    st = TileStore(T, c, Hs, Ws, device=dev, superpixels=superpixels)
    st.put(list(range(T)), soft, ids)
    return st, soft, (None if ids is None else ids[:, 0].to(torch.int32))


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


def _check(st, soft, ids, tiles, windows, Ho, Wo):
    got_s, got_i = st.batch(tiles, windows, (Ho, Wo))
    want_s, want_i = _ref(st.soft, st.ids, tiles, windows, Ho, Wo)
    assert torch.equal(got_s, want_s), (windows, Ho, Wo)
    if ids is None:
        assert got_i is None
    else:
        assert got_i.dtype == torch.int64 and got_i.shape == (len(tiles), 1, Ho, Wo)
        assert torch.equal(got_i, want_i), (windows, Ho, Wo)


@pytest.mark.gpu
@pytest.mark.parametrize("tile", [(512, 512), (1024, 1024), (97, 130)])
@pytest.mark.parametrize("c", [1, 6, 7, 8])
def test_gather_matches_torch(dev, tile, c):
    Hs, Ws = tile
    T = 5
    g = torch.Generator().manual_seed(Hs * 10 + c)
    for superpixels in (True, False):
        st, soft, ids = _filled(T, c, Hs, Ws, dev, seed=Hs + c, superpixels=superpixels)
        assert torch.equal(st.soft.cpu(), soft)
        if ids is not None:
            assert torch.equal(st.ids.cpu(), ids)
        m = min(Hs, Ws)
        calls = []
        # the full tile (a non-square tile: the transposing codes take the transposed output shape)
        calls += [(list(range(4)), Hs, Ws, "full"), (list(range(4, 8)), Ws, Hs, "full")]
        calls += [(list(range(8)), m // 2, m // 2, "odd"),            # interior crop at odd offsets
                  (list(range(8)), m - 5, m - 3, "edge"),             # touching the right and bottom edges
                  (list(range(8)), m // 2 + 3, m // 3 + 1, "any")]    # non-square window
        for codes, Ho, Wo, place in calls:
            # n = 16 with repeated tile indices (each code twice), and n = 1
            cs = codes * (16 // len(codes))
            tiles = torch.randint(0, T, (len(cs),), generator=g).tolist()
            tiles[1] = tiles[0]
            _check(st, soft, ids, tiles, _windows(cs, Hs, Ws, Ho, Wo, place, g), Ho, Wo)
            _check(st, soft, ids, [T - 1], _windows(codes[-1:], Hs, Ws, Ho, Wo, place, g), Ho, Wo)
        del st
        torch.cuda.empty_cache()


@pytest.mark.gpu
def test_store_past_2g_elements(dev):
    """c = 8, 512^2, 1100 tiles = 2.31e9 elements (9.2 GB): the last tiles lie past element 2^31."""
    T, c, H, W = 1100, 8, 512, 512
    assert T * c * H * W > 2 ** 31
    st = TileStore(T, c, H, W, device=dev)
    g = torch.Generator().manual_seed(7)
    last = list(range(T - 4, T))
    soft = torch.rand(4, c, H, W, generator=g)
    sup = torch.randint(0, 2 ** 31 - 1, (4, H, W), generator=g, dtype=torch.int64)
    st.put(last, soft.to(dev), sup.to(dev))
    assert (T - 4) * c * H * W > 2 ** 31
    codes = list(range(8))
    tiles = [last[i % 4] for i in codes]
    wins = _windows(codes, H, W, 300, 200, "any", g)
    got_s, got_i = st.batch(tiles, wins, (300, 200))
    want_s, want_i = _ref(st.soft, st.ids, tiles, wins, 300, 200)
    assert torch.equal(got_s, want_s) and torch.equal(got_i, want_i)
    # and the store really holds what was put there
    assert torch.equal(st.soft[T - 1].cpu(), soft[3]) and torch.equal(st.ids[T - 1].cpu().long(), sup[3])
    del st, got_s, got_i, want_s, want_i
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_out_of_range_samples(dev, monkeypatch):
    from uemda_b200 import config
    T, c, Hs, Ws, Ho, Wo = 4, 6, 64, 80, 32, 48
    st, soft, ids = _filled(T, c, Hs, Ws, dev, seed=3)
    good = [(0, 0, 0), (5, 7, 6), (Hs - Ho, Ws - Wo, 3)]
    bad_tiles = [(-1, (0, 0, 0)), (T, (0, 0, 0)), (2 ** 40, (0, 0, 5))]
    bad_windows = [(1, (Hs - Ho + 1, 0, 0)), (1, (0, Ws - Wo + 1, 1)), (1, (-1, 0, 2)), (1, (0, -2, 0)),
                   (1, (Hs - Wo + 1, 0, 4)), (1, (0, Ws - Ho + 1, 7)), (1, (0, 0, 8)), (1, (0, 0, -1))]
    tiles = [2, 1, 3] + [t for t, _ in bad_tiles + bad_windows]
    wins = good + [w for _, w in bad_tiles + bad_windows]
    dt = torch.tensor(tiles, dtype=torch.int64, device=dev)
    dw = torch.tensor(wins, dtype=torch.int32, device=dev)
    out = (torch.full((len(tiles), c, Ho, Wo), 7.0, device=dev), torch.full((len(tiles), 1, Ho, Wo), 7, dtype=torch.int64, device=dev))
    monkeypatch.setattr(config, "strict_asserts", False)
    got_s, got_i = st.batch(dt, dw, (Ho, Wo), out=out)
    torch.cuda.synchronize()
    assert int(st.status.item()) & 1
    want_s, want_i = _ref(st.soft, st.ids, tiles[:3], good, Ho, Wo)
    assert torch.equal(got_s[:3], want_s) and torch.equal(got_i[:3], want_i)
    assert not got_s[3:].any() and not got_i[3:].any()
    st.status.zero_()
    # a clean batch leaves the status alone; under strict_asserts a bad sample raises and the word is cleared
    st.batch(tiles[:3], good, (Ho, Wo))
    assert int(st.status.item()) == 0
    monkeypatch.setattr(config, "strict_asserts", True)
    st.batch(tiles[:3], good, (Ho, Wo))
    with pytest.raises(IndexError):
        st.batch([T], [(0, 0, 0)], (Ho, Wo))
    assert int(st.status.item()) == 0


@pytest.mark.gpu
def test_cuda_graph_replay(dev, monkeypatch):
    from uemda_b200 import config
    monkeypatch.setattr(config, "strict_asserts", False)
    T, c, Hs, Ws, Ho, Wo, n = 6, 7, 256, 256, 128, 128, 8
    st, soft, ids = _filled(T, c, Hs, Ws, dev, seed=11)
    g = torch.Generator().manual_seed(5)

    def draw():
        codes = torch.randint(0, 8, (n,), generator=g).tolist()
        return torch.randint(0, T, (n,), generator=g).tolist(), _windows(codes, Hs, Ws, Ho, Wo, "any", g)

    t0, w0 = draw()
    dt = torch.tensor(t0, dtype=torch.int64, device=dev)
    dw = torch.tensor(w0, dtype=torch.int32, device=dev)
    out = (torch.empty(n, c, Ho, Wo, device=dev), torch.empty(n, 1, Ho, Wo, dtype=torch.int64, device=dev))
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
        eager_s, eager_i = st.batch(tl, wl, (Ho, Wo))
        torch.cuda.synchronize()
        assert torch.equal(out[0], eager_s) and torch.equal(out[1], eager_i)
        want_s, want_i = _ref(st.soft, st.ids, tl, wl, Ho, Wo)
        assert torch.equal(out[0], want_s) and torch.equal(out[1], want_i)
    assert int(st.status.item()) == 0


@pytest.mark.gpu
def test_regeneration_fills_the_store(dev):
    from uemda_b200.regen import PseudoLabelRegenerator
    T, c, H, W, b = 10, 6, 64, 96, 3
    g = torch.Generator().manual_seed(9)
    soft = torch.softmax(torch.randn(T, c, H, W, generator=g), dim=1)
    sup = torch.randint(0, 50, (T, 1, H, W), generator=g, dtype=torch.int64)
    order = torch.randperm(T, generator=g).tolist()
    batches = [{"soft": soft[order[i:i + b]].pin_memory(), "sup": sup[order[i:i + b]].pin_memory(), "names": order[i:i + b],
                "tiles": order[i:i + b]} for i in range(0, T, b)]
    st = TileStore(T, c, H, W, device=dev)
    seen = []
    n = PseudoLabelRegenerator(refine=False).run(batches, lambda names, u8: seen.extend(names), device=dev, store=st)
    torch.cuda.synchronize()
    assert n == T and sorted(seen) == list(range(T))
    assert torch.equal(st.soft.cpu(), soft) and torch.equal(st.ids.cpu(), sup[:, 0].to(torch.int32))
    with pytest.raises(ValueError):
        PseudoLabelRegenerator(refine=False).run([{"soft": soft[:2]}, {"soft": soft[2:4]}], lambda *a: None, device=dev, store=st)


@pytest.mark.gpu
def test_mining_chain_on_a_gathered_batch(dev):
    """refine -> select at the cfg2 shape (8 x 6 x 512^2 out of 512^2 tiles, all 8 codes) on store.batch(...) and on the
    torch-assembled batch: bit-identical."""
    from uemda_b200 import mining, ops
    from uemda_b200.synth import WORKLOADS, make_inputs
    wl = WORKLOADS["cfg2_isprs_8x6x512"]
    inp = make_inputs(wl, with_source=False)
    st = TileStore(wl.b, wl.c, wl.H, wl.W, device=dev)
    st.put(list(range(wl.b)), inp["soft"].pin_memory(), inp["sup"].pin_memory())
    tiles = [3, 1, 4, 1, 5, 0, 2, 6]
    wins = [(0, 0, code) for code in range(8)]
    got_s, got_i = st.batch(tiles, wins, (wl.H, wl.W))
    want_s, want_i = _ref(inp["soft"].to(dev), inp["sup"][:, 0].to(dev), tiles, wins, wl.H, wl.W)
    assert torch.equal(got_s, want_s) and torch.equal(got_i, want_i)
    d = {k: inp[k].to(dev) for k in ("feat", "pred1", "pred2", "prototypes")}

    def chain(soft, sup):
        return mining.refine_select(ops.MODE_VIEWS["all"], soft, 2.0, feat=d["feat"], prototypes=d["prototypes"], pred1=d["pred1"],
                                    pred2=d["pred2"], sup=sup, select=(0.8, 0.6, -1))

    r1, h1 = chain(got_s, got_i)
    r2, h2 = chain(want_s, want_i)
    assert torch.equal(r1, r2) and torch.equal(h1, h2)


@pytest.mark.gpu
def test_gather_kernel_is_launched(dev):
    """uem_tile_gather has one kernel for every code, with and without ids."""
    import re
    from torch.profiler import ProfilerActivity, profile
    st, _, _ = _filled(2, 6, 64, 64, dev, seed=1)
    for tiles, wins in (([0, 1], [(0, 0, 0), (3, 5, 6)]), ([1], [(1, 1, 5)])):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            st.batch(tiles, wins, (40, 48))
            torch.cuda.synchronize()
        names = {e.name.replace(" ", "") for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
        assert any(re.search(r"(?<![A-Za-z0-9_])tile_gather_kernel", nm) for nm in names), sorted(names)
