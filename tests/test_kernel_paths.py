"""Every kernel an entry point can dispatch to, compared with a reference at a shape that reaches it.

Most C entry points choose between two to four kernels from the shape, the class count, the grid size and the alignment
of their pointers.  Each test here names the kernel it targets and checks, under torch.profiler, that the call launched
it, so a later change to a dispatch threshold that moves a shape onto another kernel fails instead of silently dropping
coverage.  References: the oracle where it is cheap, otherwise an exact-integer or float64 restatement in this file.
Integer outputs are bit-exact; float outputs use rtol 1e-5 with the absolute floors test_gpu_parity.py justifies.
"""
import functools
import re

import pytest
import torch

from conftest import assert_close

pytestmark = pytest.mark.gpu

RTOL = 1e-5


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from uemda_b200 import _lib
    _lib.load()  # fail loudly if the extension is missing
    return torch.device("cuda", 0)


# ------------------------------------------------------------------------------------ helpers
def _launched(fn):
    """Runs fn() under the CUDA profiler: (fn's result, names of the kernels it launched, blanks removed)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name.replace(" ", "") for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return out, names


def _ran(names, *kernels):
    """Each kernel (demangled name with its template arguments, e.g. "downscale_pow2_stream_kernel<6>") was launched."""
    for k in kernels:
        pat = re.compile(r"(?<![A-Za-z0-9_])" + re.escape(k.replace(" ", "")))
        assert any(pat.search(n) for n in names), "%s was not launched; kernels: %s" % (k, sorted(names))


def _offset(t, elems):
    """Contiguous copy of t whose data pointer sits `elems` elements past a 256-byte boundary."""
    es = t.element_size()
    buf = torch.empty(t.numel() + (256 + elems * es) // es + 1, dtype=t.dtype, device=t.device)
    start = (-buf.data_ptr() % 256) // es + elems
    v = buf[start:start + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 256 == elems * es
    return v


def _eq(a, b, what):
    a, b = a.cpu(), b.cpu()
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    bad = int((a != b).sum()) if not a.is_floating_point() else int((~((a == b) | (a.isnan() & b.isnan()))).sum())
    assert bad == 0, "%s: %d / %d elements differ" % (what, bad, a.numel())


def _lib():
    from uemda_b200 import _lib as L
    return L


# ------------------------------------------------------------------------------------ DownscaleLabel
def _cell_labels(b, h, w, s, c, seed, pad=(0, 0)):
    """(b, h*s + pad[0], w*s + pad[1]) int64 labels in [-1, c) made of whole s x s cells (the pad is random and dropped).
    Most cells are one class with a random share (0-50 %) of random labels mixed in.  When s*s % 4 == 0 a quarter are
    edge cells, each a fixed shuffle of: a majority of exactly 3/4 (rest ignore); 3/4 minus one pixel; a tie of classes
    1 and c-1; a tie of class c-1 and the ignore label; a four-way tie of 0, 1, 2 and ignore; all ignore."""
    g = torch.Generator().manual_seed(seed)
    n = s * s
    base = torch.randint(0, c, (b, h, w, 1), generator=g)
    share = torch.rand(b, h, w, 1, generator=g) * 0.5
    vals = torch.where(torch.rand(b, h, w, n, generator=g) < share, torch.randint(-1, c, (b, h, w, n), generator=g), base)
    if n % 4 == 0:
        q = n // 4
        edge = torch.full((6, n), -1, dtype=torch.int64)
        edge[0, :3 * q] = c - 1
        edge[1, :3 * q - 1] = 1
        edge[2, :2 * q] = 1
        edge[2, 2 * q:] = c - 1
        edge[3, :2 * q] = c - 1
        edge[4, :q], edge[4, q:2 * q], edge[4, 2 * q:3 * q] = 0, 1, 2
        edge = torch.stack([e[torch.randperm(n, generator=g)] for e in edge])
        kind = torch.randint(0, 24, (b, h, w), generator=g)
        vals = torch.where((kind < 6).unsqueeze(-1), edge[kind.clamp(max=5)], vals)
    lab = vals.view(b, h, w, s, s).permute(0, 1, 3, 2, 4).reshape(b, h * s, w * s)
    if pad[1]:
        lab = torch.cat([lab, torch.randint(-1, c, (b, h * s, pad[1]), generator=g)], dim=2)
    if pad[0]:
        lab = torch.cat([lab, torch.randint(-1, c, (b, pad[0], lab.shape[2]), generator=g)], dim=1)
    return lab.contiguous()


def _cell_counts(lab, s, c, ignore=-1):
    """(b, h, w, c+1) exact per-cell counts of classes 0..c-1 and (last) the ignore label; trailing rows / columns that do
    not fill a cell are dropped (alignment.py:500)."""
    b, H, W = lab.shape
    h, w = H // s, W // s
    x = lab[:, :h * s, :w * s].reshape(b, h, s, w, s)
    return torch.stack([(x == (ignore if ci == c else ci)).sum(dim=(2, 4)) for ci in range(c + 1)], dim=-1)


def _downscale_ref(cnt, s, c, min_ratio, ignore=-1):
    """alignment.py:494-509 from exact counts: first-index majority over c+1 bins, dropped when it is the ignore bin or
    its fp32 share count / (s*s) is below fp32(min_ratio) -> (b, 1, h, w)."""
    best = cnt[..., 0]
    arg = torch.zeros_like(best)
    for ci in range(1, c + 1):
        gt = cnt[..., ci] > best
        best = torch.where(gt, cnt[..., ci], best)
        arg = torch.where(gt, torch.full_like(arg, ci), arg)
    ratio = best.to(torch.float32) / float(s * s)
    low = ratio < torch.tensor(min_ratio, dtype=torch.float32)
    return torch.where((arg == c) | low, torch.full_like(arg, ignore), arg).unsqueeze(1)


@functools.lru_cache(maxsize=None)
def _downscale_case(b, h, w, s, c, pad):
    lab = _cell_labels(b, h, w, s, c, seed=b * 131 + h * 7 + s * 3 + c, pad=pad)
    return lab, _cell_counts(lab, s, c)


def _check_downscale(dev, case, s, c, kernel):
    from uemda_b200 import ops
    lab, cnt = case
    d = lab.to(dev)
    for i, mr in enumerate((0.75, 0.5, 0.25)):
        if i == 0:
            got, names = _launched(lambda: ops.downscale_label(d, s, c, -1, mr))
            _ran(names, kernel)
        else:
            got = ops.downscale_label(d, s, c, -1, mr)
        _eq(got, _downscale_ref(cnt, s, c, mr), "downscale s=%d c=%d min_ratio=%g" % (s, c, mr))


# uem_proto.cu:464: grids of more than 2 x 148 blocks take the BR = 8 stream kernel (config 3: 2048 blocks, config 5: 1024)
@pytest.mark.parametrize("b,H,W,s,c", [(16, 1024, 1024, 16, 7), (32, 512, 512, 16, 6), (8, 1024, 1024, 32, 8),
                                       (8, 512, 512, 8, 6), (8, 512, 512, 2, 3)])
def test_downscale_stream_kernel(dev, b, H, W, s, c):
    """downscale_pow2_stream_kernel at the config-3 and config-5 shapes and at s = 32, 8, 2: one, two and four 8-row load
    batches per cell, C = 8 (the ignore label counted in the separate ninth counter)."""
    _check_downscale(dev, _downscale_case(b, H // s, W // s, s, c, (0, 0)), s, c, "downscale_pow2_stream_kernel<%d>" % c)


@pytest.mark.parametrize("s", [2, 4, 8, 16, 32, 64])
@pytest.mark.parametrize("c", [3, 8])
def test_downscale_pow2_kernel(dev, s, c):
    """downscale_pow2_kernel (BR = 16) at every power-of-two scale: 1 to 32 lanes per cell (xor-shuffle folds of width 1
    to 32), one to four 16-row load batches, ties, majorities at exactly min_ratio, trailing rows / columns dropped."""
    n = max(8, 512 // s)
    pad = (s - 1, s - 2 if s > 2 else 0)
    _check_downscale(dev, _downscale_case(1, n, n, s, c, pad), s, c, "downscale_pow2_kernel<%d>" % c)


@pytest.mark.parametrize("b,h,w,s,c,pad", [(2, 16, 21, 6, 6, (5, 4)), (2, 12, 10, 12, 8, (3, 6)), (1, 8, 8, 128, 7, (0, 0)),
                                           (2, 20, 25, 3, 6, (2, 1))])
def test_downscale_generic_kernel(dev, b, h, w, s, c, pad):
    """downscale_kernel: even scales that are not powers of two (paired-column path), s = 128 (beyond the packed-counter
    limit of 64) and an odd scale (scalar path), with the same edge cells."""
    _check_downscale(dev, _downscale_case(b, h, w, s, c, pad), s, c, "downscale_kernel<%d>" % c)


# ------------------------------------------------------------------------------------ logits pass fallback
# uem_logits.cu:297: the column walk declines when its tap scratch exceeds 64 KiB, i.e. when the output is much narrower
# than the input; logits_pass_kernel<C, 4> (W % 4 == 0) or <C, 1> takes the call
@pytest.mark.parametrize("b,c,h,w,H,W,heads,temp,kernel", [
    (2, 6, 64, 300, 32, 100, 2, 1.0, "logits_pass_kernel<6, 4>"),
    (1, 6, 64, 500, 32, 101, 2, 1.7, "logits_pass_kernel<6, 1>"),
    (2, 3, 40, 1200, 20, 120, 1, 1.0, "logits_pass_kernel<3, 4>"),
    (1, 8, 16, 400, 16, 64, 2, 2.0, "logits_pass_kernel<8, 4>"),
])
def test_logits_pass_fallback_kernel(dev, b, c, h, w, H, W, heads, temp, kernel):
    from oracle import uem_oracle as O
    from uemda_b200 import ops
    g = torch.Generator().manual_seed(h * 31 + w)
    x1 = torch.randn(b, c, h, w, generator=g) * 4
    x2 = torch.randn(b, c, h, w, generator=g) * 4 if heads == 2 else None
    want = O.soft_from_logits(x1 / temp, None if x2 is None else x2 / temp, (H, W))
    out, names = _launched(lambda: ops.softmax_conf_entropy_argmax(x1.to(dev), None if x2 is None else x2.to(dev), size=(H, W),
                                                                   temp=temp))
    _ran(names, kernel)
    assert_close(out["soft"], want, rtol=RTOL, atol=1e-8, what="soft")
    conf, arg = O.confidence_argmax(want)
    assert_close(out["conf"], conf, rtol=RTOL, atol=1e-8, what="conf")
    assert_close(out["entropy"].reshape(-1), O.entropy(out["soft"].cpu()), rtol=RTOL, atol=1e-7, what="entropy of own soft")
    assert_close(out["entropy"].reshape(-1), O.entropy(want), rtol=RTOL, atol=1e-6, what="entropy")
    top2 = want.topk(2, dim=1)[0]
    clear = (top2[:, 0] - top2[:, 1]) > 1e-5
    assert bool((out["argmax"].cpu()[clear] == arg[clear]).all())
    _eq(out["argmax"], out["soft"].cpu().max(dim=1)[1], "argmax of own soft")


# ------------------------------------------------------------------------------------ prototype sums
def _proto_ref(feat, lab, c):
    """float64 masked class sums (c, k) and exact counts (c,)."""
    b, k = feat.shape[:2]
    lab = lab.reshape(b, -1)
    hot = torch.stack([(lab == ci) for ci in range(c)], dim=1).double()   # (b, c, hw); -1 matches no class
    return torch.einsum("bkn,bcn->ck", feat.reshape(b, k, -1).double(), hot), hot.sum(dim=(0, 2)).long()


def _check_proto(sums, counts, ref, what):
    want, wcnt = ref
    _eq(counts, wcnt, what + " counts")
    rms = want.pow(2).mean().sqrt().item()   # fp32 accumulation-order noise is ~3e-6 of it (test_proto_sums_benchmarked_shapes)
    assert_close(sums, want, rtol=RTOL, atol=1e-5 * rms, what=what + " sums")


# uem_proto.cu:524: hw % 4 != 0 stages the labels of an image as bytes; above 48 KiB the kernel needs the opt-in attribute
@pytest.mark.parametrize("b,k,h,w,c", [(2, 40, 223, 223, 6), (1, 33, 387, 389, 7)])
def test_proto_sums_large_label_stage(dev, b, k, h, w, c):
    from uemda_b200 import ops
    g = torch.Generator().manual_seed(h * w)
    feat = torch.randn(b, k, h, w, generator=g)
    lab = torch.randint(-1, c, (b, 1, h, w), generator=g)
    (sums, counts), names = _launched(lambda: ops.proto_accumulate(feat.to(dev), lab.to(dev), c))
    _ran(names, "proto_accum_kernel<%d, 1>" % c)
    _check_proto(sums, counts, _proto_ref(feat, lab, c), "proto sums hw=%d" % (h * w))


# ------------------------------------------------------------------------------------ Pearson k split
def _pearson_ksplit(lib, b, hw, m, k):
    """The k split of the TMA kernel, read off its workspace: [pc 8k f32][stats 2m f32][arrivals b*ptiles i32] and, when it
    splits, KS slices of (2 + m) x 128 partial sums per pixel tile (uem_pearson.cu:429)."""
    ptiles = -(-hw // 128)
    base = (((8 * k + 2 * m + 4) * 4 + 15) // 16) * 16 + ((b * ptiles * 4 + 15) // 16) * 16
    extra = lib.uem_pearson_nchw_ws_bytes(b, hw, m, k) - base
    return 1 if extra == 0 else extra // (b * ptiles * (2 + m) * 128 * 4)


@pytest.mark.parametrize("b,k,h,w,c,ks", [(4, 2048, 64, 64, 7, 2), (2, 2000, 64, 64, 6, 4), (8, 2048, 24, 30, 6, 4)])
def test_pearson_tma_ksplit(dev, b, k, h, w, c, ks):
    """KS = 2 (ptiles*b in (74, 148]); KS = 4 with k = 2000, whose last split ends in a 16-channel tile; KS = 4 with a
    partial last pixel tile (hw = 720)."""
    from oracle import uem_oracle as O
    from uemda_b200 import ops
    assert _pearson_ksplit(_lib().load(), b, h * w, c, k) == ks
    g = torch.Generator().manual_seed(k + h * w + b)
    protos = torch.randn(c, k, generator=g)
    cls = torch.randint(0, c, (b, h, w), generator=g)
    feat = (torch.randn(b, k, h, w, generator=g) + 0.5 * protos[cls].permute(0, 3, 1, 2)).contiguous()
    got, names = _launched(lambda: ops.pearson_dist_nchw(feat.to(dev), protos.to(dev)))
    _ran(names, "pearson_tma_kernel<%d>" % c)
    want = O.pearson_dist(feat.permute(0, 2, 3, 1).reshape(-1, k), protos)
    assert_close(got.permute(0, 2, 3, 1).reshape(-1, c), want, rtol=RTOL, atol=1e-6, what="pearson KS=%d" % ks)


# ------------------------------------------------------------------------------------ misaligned inputs
@functools.lru_cache(maxsize=None)
def _sweep_inputs():
    """CPU inputs at vector-eligible shapes (every width a multiple of 4)."""
    g = torch.Generator().manual_seed(2024)
    b, c, H, W, k, h, w = 2, 6, 64, 64, 64, 16, 16
    soft = torch.softmax(torch.randn(b, c, H, W, generator=g) * 3, dim=1)
    sup = (torch.arange(H).view(H, 1) // 12 * 6 + torch.arange(W).view(1, W) // 11).expand(b, 1, H, W).clone()
    sup[1] = sup[1].flip(-1)
    hard = torch.where(torch.rand(b, H, W, generator=g) < 0.2, torch.full((b, H, W), -1), soft.argmax(dim=1))
    protos = torch.randn(c, k, generator=g)
    feat = torch.randn(b, k, h, w, generator=g) + 0.5 * protos[torch.randint(0, c, (b, h, w), generator=g)].permute(0, 3, 1, 2)
    return dict(
        soft=soft, sup=sup, hard=hard, feat=feat.contiguous(), protos=protos,
        pred1=torch.randn(b, c, h, w, generator=g) * 4, pred2=torch.randn(b, c, h, w, generator=g) * 4,
        label_low=torch.randint(-1, c, (b, 1, h, w), generator=g),
        label_full=_cell_labels(b, H * 4 // 16, W * 4 // 16, 16, c, seed=5),   # (2, 256, 256): the pow2 kernel at s = 16
        table=torch.rand(c, generator=g) + 0.1,
    )


def _run_select(x):
    from uemda_b200 import ops
    cmax, cmin, nan = ops.class_max(x["soft"])
    return cmax, cmin, nan, ops.pseudo_select(x["soft"], cmax, 0.8, 0.6)


def _run_entropy(x):
    from uemda_b200 import ops
    return ops.entropy_uvem_weight(x["soft"], 0.2, 0.7, 4.0)


def _run_uvem_terms(x):
    from uemda_b200 import ops
    return ops.uvem_terms(x["soft"], x["hard"], 0.2, 0.7, 4.0)


def _run_downscale(x):
    from uemda_b200 import ops
    return (ops.downscale_label(x["label_full"], 16, 6),)


def _run_region(red):
    def run(x):
        from uemda_b200 import ops
        return (ops.region_reduce(x["soft"], x["sup"], red, planar=True),)
    return run


def _ref_region(red):
    def ref(x):
        from oracle import uem_oracle as O
        b, c = x["soft"].shape[:2]
        rows = x["soft"].permute(0, 2, 3, 1).reshape(b, -1, c)
        return (O.region_reduce(rows.double(), x["sup"].reshape(b, -1, 1), red).float(),)
    return ref


def _run_expand(x):
    from uemda_b200 import ops
    return (ops.superpixel_expand(x["hard"], x["sup"], 6),)


def _run_pearson(x):
    from uemda_b200 import ops
    return (ops.pearson_dist_nchw(x["feat"], x["protos"]),)


def _ref_pearson(x):
    from oracle import uem_oracle as O
    b, k, h, w = x["feat"].shape
    return (O.pearson_dist(x["feat"].permute(0, 2, 3, 1).reshape(-1, k), x["protos"]).reshape(b, h, w, -1).permute(0, 3, 1, 2),)


def _run_proto(x):
    from uemda_b200 import ops
    return ops.proto_accumulate(x["feat"], x["label_low"], 6)


def _run_class_hist(x):
    from uemda_b200 import ops
    return (ops.class_hist(x["hard"], 6),)


def _run_weight_lookup(x):
    from uemda_b200 import ops
    return (ops.class_weight_lookup(x["hard"], x["table"]),)


def _run_plus1(x):
    from uemda_b200 import ops
    return (ops.label_plus1_u8(x["hard"]),)


def _run_iast(x):
    from uemda_b200.utils.tools import IASTSelector
    sel = IASTSelector(n_class=6, pl_alpha=0.2, pl_beta=0.9, pl_gamma=8.0, device=x["soft"].device)
    labels = sel.step(x["soft"])
    return labels, sel.cls_thresh, sel.tmp_thresh, sel.counts


def _run_refine(x):
    from uemda_b200 import mining
    refined, _ = mining.refine_select(7, x["soft"], 2.0, feat=x["feat"], prototypes=x["protos"], pred1=x["pred1"],
                                      pred2=x["pred2"], sup=x["sup"])
    return (refined,)


def _ref_refine(x):
    from oracle import uem_oracle as O
    return (O.label_refine(x["sup"], x["feat"], [x["pred1"], x["pred2"]], x["soft"], x["protos"], mode="all", temp=2.0),)


# name -> (run, inputs to misalign, kernels of the aligned call, kernels of the misaligned call, reference or None).
# None: the vector and the scalar kernel do the same arithmetic in the same order, so the misaligned call must be
# bit-identical to the aligned one.  A reference is given where the two kernels sum in different orders (Pearson, the
# prototype sums, the refine kernels) or where float atomics make the order run-dependent (region sum / mean).
SWEEP = {
    "select": (_run_select, ["soft"], ["class_max_partial_kernel<4>", "select_kernel<6, 4>"],
               ["class_max_partial_kernel<1>", "select_kernel<6, 1>"], None),
    "entropy_uvem": (_run_entropy, ["soft"], ["entropy_weight_kernel<6, 4, false>"], ["entropy_weight_kernel<6, 1, false>"], None),
    "uvem_terms_soft": (_run_uvem_terms, ["soft"], ["entropy_weight_kernel<6, 4, true>"], ["entropy_weight_kernel<6, 1, true>"], None),
    "uvem_terms_target": (_run_uvem_terms, ["hard"], ["entropy_weight_kernel<6, 4, true>"], ["entropy_weight_kernel<6, 1, true>"],
                          None),
    "downscale": (_run_downscale, ["label_full"], ["downscale_pow2_kernel<6>"], ["downscale_kernel<6>"], None),
    "region_max_src": (_run_region("max"), ["soft"], ["region_max_smem_kernel<6, 4>"], ["region_max_smem_kernel<6, 1>"], None),
    "region_max_index": (_run_region("max"), ["sup"], ["region_max_smem_kernel<6, 4>"], ["region_max_smem_kernel<6, 1>"], None),
    "region_sum_src": (_run_region("sum"), ["soft"], ["region_reduce_f32_kernel<6, 4"], ["region_reduce_f32_kernel<6, 1"],
                       _ref_region("sum")),
    "region_mean_index": (_run_region("mean"), ["sup"], ["region_reduce_f32_kernel<6, 4"], ["region_reduce_f32_kernel<6, 1"],
                          _ref_region("mean")),
    "expand_hard": (_run_expand, ["hard"], ["region_hist_smem_kernel<6, 4>", "region_gather_label_kernel<4>"],
                    ["region_class_hist_kernel<6, 1>", "region_gather_label_kernel<1>"], None),
    "expand_sup": (_run_expand, ["sup"], ["region_hist_smem_kernel<6, 4>", "region_gather_label_kernel<4>"],
                   ["region_class_hist_kernel<6, 1>", "region_gather_label_kernel<1>"], None),
    "pearson": (_run_pearson, ["feat"], ["pearson_tma_kernel<6>"], ["pearson_nchw_kernel<6, 1>"], _ref_pearson),
    "proto_feat": (_run_proto, ["feat"], ["proto_accum_tma_kernel<6, 4>"], ["proto_accum_kernel<6, 1>"], "proto"),
    "proto_label": (_run_proto, ["label_low"], ["proto_accum_tma_kernel<6, 4>"], ["proto_accum_kernel<6, 1>"], "proto"),
    "class_hist": (_run_class_hist, ["hard"], ["class_hist_kernel<6>"], ["class_hist_kernel<6>"], None),
    "weight_lookup": (_run_weight_lookup, ["hard"], ["class_weight_lookup_kernel"], ["class_weight_lookup_kernel"], None),
    "label_plus1": (_run_plus1, ["hard"], ["label_plus1_u8_kernel"], ["label_plus1_u8_kernel"], None),
    "iast": (_run_iast, ["soft"], ["iast_hist_kernel<6, 4>", "iast_label_kernel<6, 4>"],
             ["iast_hist_kernel<6, 1>", "iast_label_kernel<6, 1>"], None),
    "refine_soft": (_run_refine, ["soft"], ["refine_col_kernel<6"], ["refine_kernel<6, 1>"], _ref_refine),
    "refine_sup": (_run_refine, ["sup"], ["refine_col_kernel<6"], ["refine_kernel<6, 1>"], _ref_refine),
}


@pytest.mark.parametrize("off", [1, 3])
@pytest.mark.parametrize("case", list(SWEEP))
def test_misaligned_inputs(dev, case, off):
    """Each input a vector kernel reads in 16-byte accesses, handed over `off` elements past a 256-byte boundary
    (L.f32c / L.i64c accept any contiguous view): the call must take the scalar kernel and give the aligned result.
    proto_label is the regression test of the prototype sums, which used to read a misaligned label map with the TMA
    kernel's 16-byte loads."""
    run, moved, vec_kernels, scalar_kernels, ref = SWEEP[case]
    cpu = _sweep_inputs()
    aligned = {key: t.to(dev) for key, t in cpu.items()}
    shifted = dict(aligned, **{key: _offset(aligned[key], off) for key in moved})
    want, names = _launched(lambda: run(aligned))
    _ran(names, *vec_kernels)
    got, names = _launched(lambda: run(shifted))
    _ran(names, *scalar_kernels)
    if ref is None:
        for i, (a, b) in enumerate(zip(got, want)):
            _eq(a, b, "%s output %d, offset %d vs aligned" % (case, i, off))
    elif ref == "proto":
        r = _proto_ref(cpu["feat"], cpu["label_low"], 6)
        _check_proto(*want, r, "aligned")
        _check_proto(*got, r, "offset %d" % off)
    else:
        r = ref(cpu)
        for out, what in ((want, "aligned"), (got, "offset %d" % off)):
            for a, b in zip(out, r):
                assert_close(a, b, rtol=RTOL, atol=1e-6, what="%s %s" % (case, what))


@pytest.mark.parametrize("arg", ["feat", "coef", "grad"])
def test_pcl_refuses_misaligned_maps(dev, arg):
    """The contrastive-loss kernels stream the feature map through TMA and have no scalar form: they refuse a
    misaligned map with an error instead of reading it."""
    from uemda_b200 import _lib as L, ops
    g = torch.Generator().manual_seed(3)
    feat = torch.randn(2, 64, 8, 8, generator=g).to(dev)
    protos = torch.randn(6, 64, generator=g).to(dev)
    labels = torch.randint(-1, 6, (2, 8, 8), generator=g).to(dev)
    if arg == "feat":
        with pytest.raises(L.UemLibraryError, match="16-byte aligned"):
            ops.pcl_forward(_offset(feat, 1), protos, labels)
        return
    loss, coef, ws = ops.pcl_forward(feat, protos, labels)
    lib = L.load()
    grad = torch.empty_like(feat)
    if arg == "coef":
        coef = _offset(coef, 1)
    else:
        grad = _offset(grad, 1)
    rc = lib.uem_pcl_backward_f32(L.ptr(feat), 2, 64, 64, 6, L.ptr(coef), None, L.ptr(grad), L.ptr(ws), L.stream_of(feat))
    assert rc != 0 and b"16-byte aligned" in lib.uem_last_error()


# ------------------------------------------------------------------------------------ entry points without a test of their own
def _labels_with_tail(n, c, seed):
    """int64 labels in [-3, c + 2) (ignore and out of range included); the last 8 are valid classes."""
    g = torch.Generator().manual_seed(seed)
    lab = torch.randint(-3, c + 2, (n,), generator=g)
    lab[-8:] = torch.randint(0, c, (8,), generator=g)
    return lab


@pytest.mark.parametrize("n", [4096, 4097, 4099])
@pytest.mark.parametrize("moved", [None, "label", "out"])
def test_class_weight_lookup_paths(dev, n, moved):
    """The 4-wide body, the n % 4 tail and the scalar path (misaligned label or output map); ignored and out-of-range
    labels weigh 0 (balance.py:29-32).  The output starts as NaN, so an element the kernel skips fails."""
    L = _lib()
    lib = L.load()
    c = 6
    lab = _labels_with_tail(n, c, seed=n)
    table = torch.rand(c) + 0.1
    valid = (lab >= 0) & (lab < c)
    want = torch.where(valid, table[lab.clamp(0, c - 1)], torch.zeros(n))
    d = lab.to(dev)
    out = torch.full((n,), float("nan"), device=dev)
    if moved == "label":
        d = _offset(d, 1)
    elif moved == "out":
        out = _offset(out, 1)
    tab = table.to(dev)
    _, names = _launched(lambda: L.check(lib.uem_class_weight_lookup_f32(L.ptr(d), n, c, -1, L.ptr(tab), L.ptr(out), L.stream_of(d))))
    _ran(names, "class_weight_lookup_kernel")
    _eq(out, want, "class weight lookup n=%d moved=%s" % (n, moved))


@pytest.mark.parametrize("n", [4096, 4097, 4098, 4099])
@pytest.mark.parametrize("moved", [None, "label", "out"])
def test_label_plus1_paths(dev, n, moved):
    """uint8(label + 1) (pseudo_generation.py:150-151) through the 4-labels-per-store body, the n % 4 tail and the scalar
    path; labels outside [-1, 254] wrap mod 256.  Run over two different initial outputs, so a skipped element fails."""
    L = _lib()
    lib = L.load()
    g = torch.Generator().manual_seed(n)
    lab = torch.randint(-1, 255, (n,), generator=g)
    lab[:8] = torch.tensor([255, -2, 1000, -300, 2 ** 40 + 7, -(2 ** 40) - 1, 254, -1])
    want = ((lab + 1) & 255).to(torch.uint8)
    d = lab.to(dev)
    if moved == "label":
        d = _offset(d, 1)
    for fill in (0, 255):
        out = torch.full((n,), fill, dtype=torch.uint8, device=dev)
        if moved == "out":
            out = _offset(out, 1)
        _, names = _launched(lambda: L.check(lib.uem_label_plus1_u8_i64(L.ptr(d), n, L.ptr(out), L.stream_of(d))))
        _ran(names, "label_plus1_u8_kernel")
        _eq(out, want, "label_plus1 n=%d moved=%s fill=%d" % (n, moved, fill))


def test_region_reduce_i64_max_of_negative_values(dev):
    """Integer region max over values that are all negative: the INT64_MIN fill and region_finish_i64_kernel, which turns
    untouched slots into 0 (torch_scatter's fill) and leaves every real maximum, however negative, alone."""
    from oracle import uem_oracle as O
    from uemda_b200 import ops
    g = torch.Generator().manual_seed(9)
    b, N, c, R = 2, 5000, 3, 40
    idx = torch.randint(0, R - 8, (b, N), generator=g)       # ids R-8 .. R-1 stay empty
    idx[:, ::7] = 5                                           # a crowded id
    src = -torch.randint(1, 1 << 40, (b, N, c), generator=g)
    got, names = _launched(lambda: ops.region_reduce(src.to(dev), idx.to(dev), "max", dim_size=R))
    _ran(names, "region_reduce_i64_kernel", "region_finish_i64_kernel")
    want = O.region_reduce(src, idx.reshape(b, N, 1), "max", dim_size=R)
    assert bool((want[:, :R - 8] < 0).all()) and bool((want[:, R - 8:] == 0).all())
    _eq(got, want, "region max i64")
    _eq(ops.region_reduce(src.to(dev), idx.to(dev), "sum", dim_size=R), O.region_reduce(src, idx.reshape(b, N, 1), "sum", dim_size=R),
        "region sum i64")


@pytest.mark.parametrize("off", [0, 1, 3])
@pytest.mark.parametrize("n", [100003, 100000, 1])
def test_i64_minmax(dev, n, off):
    """[min, max] of negative int64 values, aligned (pairs of 16-byte loads + the odd last element) and misaligned (scalar)."""
    from uemda_b200 import ops
    g = torch.Generator().manual_seed(n)
    x = -torch.randint(1, 1 << 50, (n,), generator=g)
    x[-1] = -(1 << 60)            # the minimum sits in the element a pair loop leaves over when n is odd
    if n > 2:
        x[n // 2] = -1            # the maximum
    d = x.to(dev)
    if off:
        d = _offset(d, off)
    got, names = _launched(lambda: ops.i64_minmax(d))
    _ran(names, "minmax_kernel")
    _eq(got, torch.stack([x.min(), x.max()]), "minmax n=%d off=%d" % (n, off))


@pytest.mark.parametrize("bins,lo,hi", [(30, 0.0, 1.0), (7, -0.3, 1.7), (100, 0.0, 1.0), (3, 1.0, 2.0)])
def test_hist_f32_bin_edges(dev, bins, lo, hi):
    """torch.histc exactly on the bin edges (three fp32 forms of lo + i * (hi - lo) / bins), one ulp either side of them,
    at x == lo and x == hi (last bin), just outside [lo, hi] and at NaN (dropped).  torch bins by (x - lo) * bins / (hi - lo)
    alone, so a value on a computed edge may land one bin below it."""
    from uemda_b200 import ops
    lo, hi = ops.f32(lo), ops.f32(hi)
    i = torch.arange(bins + 1, dtype=torch.float64)
    edges = torch.cat([torch.linspace(lo, hi, bins + 1, dtype=torch.float32),
                       (lo + i * ((hi - lo) / bins)).float(),
                       torch.tensor(lo, dtype=torch.float32) + torch.arange(bins + 1, dtype=torch.float32) *
                       ((torch.tensor(hi, dtype=torch.float32) - lo) / bins)])
    x = torch.cat([edges, torch.nextafter(edges, torch.tensor(float("inf"))), torch.nextafter(edges, torch.tensor(float("-inf"))),
                   torch.tensor([lo, hi, hi, float("nan")], dtype=torch.float32)])
    got, names = _launched(lambda: ops.hist_f32(x.to(dev), bins, lo, hi))
    _ran(names, "hist_f32_kernel")
    _eq(got, torch.histc(x, bins, lo, hi).long(), "histc bins=%d [%g, %g]" % (bins, lo, hi))
