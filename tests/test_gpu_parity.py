"""GPU parity: the CUDA path (through the C-ABI, via the drop-in Python layer) against
  (1) the committed golden fixtures = outputs of the reference itself (tests/golden, oracle/gen_golden.py),
  (2) the CPU oracle (oracle/uem_oracle.py) on seeded synthetic inputs.
Integer / index outputs must be bit-exact; float outputs within rtol 1e-5 (the north_star tolerance).
"""
import numpy as np
import pytest
import torch

from conftest import assert_close

pytestmark = pytest.mark.gpu

RTOL = 1e-5  # north_star: "within 1e-5 relative for entropy, thresholds and prototypes"


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from uemda_b200 import _lib
    _lib.load()  # fail loudly if the extension is missing
    return torch.device("cuda", 0)


class _Log:
    def info(self, *a, **k):
        pass


def _aligner(g, dev, protos=None):
    from uemda_b200.gast.alignment import Aligner, DownscaleLabel
    al = Aligner(_Log(), feat_channels=g.k, class_num=g.c, ignore_label=-1, decay=g.decay)
    al.downscale_gt = DownscaleLabel(scale_factor=g.scale, n_classes=g.c, ignore_label=-1, min_ratio=0.75)
    al.prototypes = (g.t("in_prototypes") if protos is None else protos).to(dev)
    return al


def _eq(a, b, what):
    a, b = a.cpu(), b.cpu()
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    bad = int((a != b).sum())
    assert bad == 0, "%s: %d / %d elements differ" % (what, bad, a.numel())


# ------------------------------------------------------------------------------------ golden fixtures
def test_golden_selection_bit_exact(golden, dev):
    from uemda_b200.gast.pseudo_generation import pseudo_selection, pseudo_selection1
    g = golden
    soft, refined = g.t("in_soft", dev), g.t("out_refine_all", dev)
    _eq(pseudo_selection(refined, 0.8, 0.6, "tensor", -1), g.t("out_select_refined"), "select refined")
    _eq(pseudo_selection(soft, 0.8, 0.6, "tensor", -1), g.t("out_select_soft"), "select soft")
    _eq(pseudo_selection(soft, 0.5, 0.2, "tensor", -1), g.t("out_select_soft_lowcut"), "select lowcut")
    _eq(pseudo_selection1(soft, 0.8, 0.6, "tensor", -1), g.t("out_select1_soft"), "select v1")
    nd = pseudo_selection(soft)
    assert isinstance(nd, np.ndarray) and nd.dtype == np.int64
    assert (nd == g.z["out_select_soft"]).all()


def test_golden_expand_downscale_bit_exact(golden, dev):
    g = golden
    al = _aligner(g, dev)
    hard = g.t("out_select_soft", dev)
    _eq(al.superpixel_expand(hard, g.t("in_sup", dev)), g.t("out_expand"), "superpixel_expand")
    _eq(al.downscale_gt(g.t("in_label_s", dev)), g.t("out_downscale_src"), "downscale src")
    _eq(al.downscale_gt(hard), g.t("out_downscale_hard"), "downscale hard")
    _eq(al.downscale_gt(hard.unsqueeze(1)), g.t("out_downscale_hard"), "downscale hard 4d")


def test_golden_pearson(golden, dev):
    g = golden
    al = _aligner(g, dev)
    flat = g.t("in_feat", dev).permute(0, 2, 3, 1).reshape(-1, g.k)
    got = al._pearson_dist(flat, al.prototypes)
    assert_close(got, g.t("out_pearson"), rtol=RTOL, atol=1e-6, what="pearson rows")
    from uemda_b200 import ops
    nchw = ops.pearson_dist_nchw(g.t("in_feat", dev), al.prototypes)
    want = g.t("out_pearson").reshape(g.b, g.H // g.scale, g.W // g.scale, g.c).permute(0, 3, 1, 2)
    assert_close(nchw, want, rtol=RTOL, atol=1e-6, what="pearson nchw")


@pytest.mark.parametrize("mode", ["all", "s", "p", "l"])
def test_golden_label_refine(golden, dev, mode):
    g = golden
    al = _aligner(g, dev)
    preds = [p.to(dev) for p in g.preds()] if g.two_heads else g.preds().to(dev)
    got = al.label_refine(g.t("in_sup", dev), g.t("in_feat", dev), preds, g.t("in_soft", dev), refine=True, mode=mode, temp=2.0)
    assert_close(got, g.t("out_refine_" + mode), rtol=RTOL, atol=1e-7, what="label_refine " + mode)
    soft = g.t("in_soft", dev)
    assert al.label_refine(g.t("in_sup", dev), g.t("in_feat", dev), preds, soft, refine=False) is soft


def test_golden_refine_then_select_chain(golden, dev):
    """End to end: refined map from the CUDA path -> selection; labels may differ from the reference only
    where a refined probability sits within float tolerance of its threshold."""
    from uemda_b200.gast.pseudo_generation import pseudo_selection
    g = golden
    al = _aligner(g, dev)
    preds = [p.to(dev) for p in g.preds()] if g.two_heads else g.preds().to(dev)
    refined = al.label_refine(g.t("in_sup", dev), g.t("in_feat", dev), preds, g.t("in_soft", dev), mode="all", temp=2.0)
    hard = pseudo_selection(refined, 0.8, 0.6, "tensor", -1)
    want = g.t("out_select_refined")
    mism = int((hard.cpu() != want).sum())
    assert mism <= max(1, want.numel() // 20000), "end-to-end label mismatches: %d of %d" % (mism, want.numel())
    # cached-partials path and the plain two-pass path must agree exactly
    _eq(pseudo_selection(refined.clone(), 0.8, 0.6, "tensor", -1), hard, "partials vs two-pass")


def test_golden_prototypes(golden, dev):
    g = golden
    al = _aligner(g, dev)
    down = al.update_prototype(g.t("in_feat_s", dev), g.t("in_label_s", dev))
    _eq(down, g.t("out_update_down"), "update_prototype down")
    assert_close(al.prototypes, g.t("out_proto_after1"), rtol=RTOL, atol=1e-7, what="proto after 1")
    local = al._compute_local_prototypes(g.t("in_feat_s", dev), down, update=False)
    assert_close(local, g.t("out_local_proto"), rtol=RTOL, atol=1e-7, what="local proto")
    al.update_prototype(g.t("in_feat", dev), g.t("in_label_s", dev))
    assert_close(al.prototypes, g.t("out_proto_after2"), rtol=RTOL, atol=1e-7, what="proto after 2")
    al.update_prototype_bytarget(g.t("in_feat", dev), g.t("in_soft", dev))
    assert_close(al.prototypes, g.t("out_proto_bytarget"), rtol=RTOL, atol=1e-7, what="proto bytarget")
    al.update_avg(g.t("in_feat_s", dev), g.t("in_label_s", dev))
    al.update_avg(g.t("in_feat", dev), g.t("in_label_s", dev))
    assert_close(al._data_sum, g.t("out_avg_sum"), rtol=RTOL, atol=1e-5, what="avg sum")
    _eq(al._data_cnt, g.t("out_avg_cnt"), "avg cnt")
    al.init_avg()
    assert_close(al.prototypes, g.t("out_avg_proto"), rtol=RTOL, atol=1e-7, what="avg proto")


def test_golden_proto_weight_4pixel(golden, dev):
    g = golden
    al = _aligner(g, dev)
    got = al.get_prototype_weight_4pixel(g.t("in_feat", dev), g.t("out_select_soft", dev))
    assert_close(got, g.t("out_proto_weight_4pixel"), rtol=RTOL, atol=1e-7, what="proto weight 4pixel")


def test_golden_logits_entropy_weight(golden, dev):
    from uemda_b200 import ops
    from uemda_b200.gast.balance import UVEMLoss
    g = golden
    out = ops.softmax_conf_entropy_argmax(g.t("in_pred1", dev), g.t("in_pred2", dev), size=(g.H, g.W))
    want = g.t("out_soft_from_logits")
    assert_close(out["soft"], want, rtol=RTOL, atol=1e-8, what="soft from logits")
    conf, arg = want.max(dim=1)
    assert_close(out["conf"], conf, rtol=RTOL, atol=1e-8, what="conf")
    # argmax may legitimately differ only where the top two classes tie within float tolerance
    top2 = want.topk(2, dim=1)[0]
    clear = (top2[:, 0] - top2[:, 1]) > 1e-5
    assert bool((out["argmax"].cpu()[clear] == arg[clear]).all())
    refined = g.t("out_refine_all", dev)
    ent, wgt = ops.entropy_uvem_weight(refined, 0.2, 0.7, 4.0)
    assert_close(ent, g.t("out_entropy"), rtol=RTOL, atol=1e-7, what="entropy")
    fn = UVEMLoss(m=0.2, threshold=0.7, gamma=4.0, class_num=g.c)
    # weight from the reference's own entropy values: isolates get_weight
    assert_close(fn.get_weight(g.t("out_entropy", dev)), g.t("out_uvem_weight"), rtol=RTOL, atol=1e-6, what="uvem weight")
    assert_close(fn.get_weight(g.t("in_uvem_grid", dev)), g.t("out_uvem_weight_grid"), rtol=RTOL, atol=1e-6, what="uvem grid")


def test_golden_class_balance_and_losses(golden, dev):
    from uemda_b200.gast.balance import ClassBalance, UPSLoss, UVEMLoss
    g = golden
    cb = ClassBalance(class_num=g.c, ignore_label=-1, decay=0.99, temperature=0.5)
    hard_r, hard = g.t("out_select_refined", dev), g.t("out_select_soft", dev)
    w1 = cb.get_class_weight_4pixel(hard_r.reshape(-1))
    assert_close(w1, g.t("out_cb_weight1"), rtol=RTOL, atol=1e-7, what="cb weight 1")
    assert_close(cb.freq, g.t("out_cb_freq1"), rtol=RTOL, atol=1e-8, what="cb freq 1")
    w2 = cb.get_class_weight_4pixel(hard.reshape(-1))
    assert_close(w2, g.t("out_cb_weight2"), rtol=RTOL, atol=1e-7, what="cb weight 2")
    assert_close(cb.freq, g.t("out_cb_freq2"), rtol=RTOL, atol=1e-8, what="cb freq 2")
    fn = UVEMLoss(m=0.2, threshold=0.7, gamma=4.0, class_balancer=cb, class_num=g.c, ignore_label=-1)
    logits = g.t("in_logits", dev).clone().requires_grad_(True)
    loss = fn(logits, hard_r, g.t("out_refine_all", dev))
    loss.backward()
    assert_close(loss.reshape(1), g.t("out_uvem_loss"), rtol=1e-4, atol=1e-6, what="uvem loss")
    assert_close(logits.grad.abs().sum().reshape(1), g.t("out_uvem_loss_grad_sum"), rtol=1e-4, atol=1e-6, what="uvem grad")
    assert_close(cb.freq, g.t("out_cb_freq3"), rtol=RTOL, atol=1e-8, what="cb freq 3")
    ups = UPSLoss(threshold=0.7, class_num=g.c)
    assert_close(ups(g.t("in_logits", dev), hard_r, g.t("out_refine_all", dev)).reshape(1), g.t("out_ups_loss"),
                 rtol=1e-4, atol=1e-6, what="ups loss")


def test_golden_scatter_seam(golden, dev):
    from uemda_b200.scatter import scatter
    g = golden
    rows = g.t("in_soft", dev).permute(0, 2, 3, 1).reshape(g.b, -1, g.c).contiguous()
    idx = g.t("in_sup", dev).reshape(g.b, -1, 1)
    _eq(scatter(rows, idx, dim=1, reduce="max"), g.t("out_scatter_max"), "scatter max")


def test_edge_cases(edge_cases, dev):
    from uemda_b200 import ops
    from uemda_b200.gast.balance import UVEMLoss
    from uemda_b200.gast.pseudo_generation import pseudo_selection, pseudo_selection1
    e = edge_cases
    p = e.t("in_prob", dev)
    ent, wgt = ops.entropy_uvem_weight(p, 0.2, 0.7, 4.0)
    assert_close(ent, e.t("out_entropy"), rtol=RTOL, atol=1e-7, what="edge entropy (NaN pattern must match)")
    assert_close(wgt, e.t("out_weight"), rtol=RTOL, atol=1e-6, what="edge weight")
    _eq(pseudo_selection(p, 0.8, 0.6, "tensor", -1), e.t("out_select"), "edge select")
    _eq(pseudo_selection1(p, 0.8, 0.6, "tensor", -1), e.t("out_select1"), "edge select1")
    for key in [k for k in e.z.files if k.startswith("in_u_")]:
        m, t, gm = [float(v) for v in key[5:].split("_")]
        fn = UVEMLoss(m=m, threshold=t, gamma=gm)
        assert_close(fn.get_weight(e.t(key, dev)), e.t("out_w_" + key[5:]), rtol=RTOL, atol=1e-6, what=key)
    with pytest.raises(AssertionError):
        pseudo_selection(p * 1.5, 0.8, 0.6, "tensor", -1)  # range assert, pseudo_generation.py:71
    with pytest.raises(RuntimeError):
        from uemda_b200.gast.alignment import DownscaleLabel
        DownscaleLabel(4, 6)(torch.full((1, 8, 8), 9, dtype=torch.int64, device=dev))  # one_hot rejects class 9


# ------------------------------------------------------------------------------------ oracle on seeded inputs
def _to(inp, dev):
    return {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in inp.items()}


@pytest.mark.parametrize("name,b,shrink", [("cfg1_cpu_2x6x512", 2, True), ("cfg3_loveda_16x7x1024", 1, True),
                                           ("cfg2_isprs_8x6x512_os8", 1, True), ("cfg1_cpu_2x6x512", 1, False)])
def test_oracle_mining_step(dev, name, b, shrink):
    """Whole step at BASELINE config shapes (batch trimmed so the CPU oracle stays in seconds).  shrink=False: the
    superpixel maps without the 7x7 edge shrink (SURVEY section 8d): no pixel carries the ignore id, so the batch max id
    that alignment.py:241 treats as "ignored" is a REAL region."""
    from oracle import uem_oracle as O
    from uemda_b200 import mining, ops
    from uemda_b200.gast.alignment import Aligner, DownscaleLabel
    from uemda_b200.synth import WORKLOADS, make_inputs
    wl = WORKLOADS[name]
    k = 256  # oracle cost is linear in k; the kernels' k loop is exercised at 2048 in test_full_size_properties
    wl = type(wl)(wl.name, b, wl.c, wl.H, wl.W, k, wl.scale, wl.regions)
    inp = make_inputs(wl, seed=7, shrink=shrink)
    want = O.mining_step(inp, inp["prototypes"], wl.c, scale_factor=wl.scale)
    d = _to(inp, dev)
    al = Aligner(_Log(), feat_channels=k, class_num=wl.c, decay=0.996)
    al.downscale_gt = DownscaleLabel(wl.scale, wl.c, -1, 0.75)
    al.prototypes = d["prototypes"].clone()
    refined, hard = mining.mine_step(al, d["sup"], d["feat"], [d["pred1"], d["pred2"]], d["soft"])
    assert_close(refined, want["refined"], rtol=RTOL, atol=1e-7, what="refined")
    mism = int((hard.cpu() != want["hard"]).sum())
    assert mism <= max(2, want["hard"].numel() // 50000), "label mismatches %d" % mism
    # bit-exact selection given the identical (oracle) refined map
    from uemda_b200.gast.pseudo_generation import pseudo_selection
    _eq(pseudo_selection(want["refined"].to(dev), 0.8, 0.6, "tensor", -1), want["hard"], "select on oracle refined")
    down = al.update_prototype(d["feat_s"], d["label_s"])
    _eq(down, want["label_s_down"], "downscale")
    assert_close(al.prototypes, want["prototypes"], rtol=RTOL, atol=1e-7, what="prototypes")
    ent, wgt = ops.entropy_uvem_weight(want["refined"].to(dev), 0.2, 0.7, 4.0)
    assert_close(ent, want["entropy"], rtol=RTOL, atol=1e-7, what="entropy")
    # get_weight on the oracle's own entropy: 1e-5.  The fused entropy->weight output inherits the entropy's 1e-5
    # through w = x^(1/gamma), whose slope is unbounded at x -> 0 (u -> threshold): absolute tolerance there.
    from uemda_b200.gast.balance import UVEMLoss
    fn = UVEMLoss(m=0.2, threshold=0.7, gamma=4.0, class_num=wl.c)
    assert_close(fn.get_weight(want["entropy"].to(dev)), want["uvem_weight"], rtol=RTOL, atol=1e-6, what="uvem weight")
    # the fused weight sees the kernel's OWN entropy (1e-5 relative): its tolerance is that error times the local slope
    # |dw/du| of w = x^(1/gamma), x = coef (u - m)^2 + 1 (balance.py:396-423), instead of one loose bound for every pixel
    m_, t_, ig, cl, cr = [float(v) for v in ops._uvem_coefs(0.2, 0.7, 4.0)]
    u = want["entropy"].double().flatten()
    coef = torch.where(u <= m_, torch.full_like(u, cl), torch.full_like(u, cr))
    x = (coef * (u - m_) ** 2 + 1.0).clamp(1e-12, 1.0)
    slope = ig * x ** (ig - 1.0) * 2.0 * coef.abs() * (u - m_).abs()
    tol = 2.0 * slope * (1e-5 * u.abs() + 1e-7) + 2e-6
    tol = torch.where((u - t_).abs() <= 2e-5 * t_, torch.full_like(tol, 0.15), tol)   # the gate u >= t itself: w jumps to 0
    err = (wgt.detach().cpu().double().flatten() - want["uvem_weight"].double().flatten()).abs()
    bad = ~((err <= tol) | (torch.isnan(u) & torch.isnan(wgt.detach().cpu().double().flatten())))
    assert not bool(bad.any()), "fused entropy->uvem weight: %d pixels beyond the propagated 1e-5 (worst %.3g at tol %.3g)" % (
        int(bad.sum()), float(err[bad].max()), float(tol[bad][err[bad].argmax()]))
    exp = al.superpixel_expand(want["hard"].to(dev), d["sup"])
    _eq(exp, O.superpixel_expand(want["hard"], inp["sup"], wl.c), "expand")


@pytest.mark.parametrize("shape", [(1, 3, 17, 23), (2, 5, 33, 64), (1, 8, 40, 36), (3, 2, 16, 20)])
def test_ragged_shapes_scalar_path(dev, shape):
    """Odd widths / unaligned views force the scalar (VEC=1) kernels."""
    from oracle import uem_oracle as O
    from uemda_b200 import ops
    from uemda_b200.gast.pseudo_generation import pseudo_selection, pseudo_selection1
    b, c, H, W = shape
    g = torch.Generator().manual_seed(b * 1000 + W)
    soft = torch.softmax(torch.randn(b, c, H, W, generator=g) * 3, dim=1)
    _eq(pseudo_selection(soft.to(dev), 0.8, 0.6, "tensor", -1), O.pseudo_select(soft), "select ragged")
    _eq(pseudo_selection1(soft.to(dev), 0.7, 0.3, "tensor", -5), O.pseudo_select_v1(soft, 0.7, 0.3, -5), "select1 ragged")
    sup = torch.randint(0, 7, (b, 1, H, W), generator=g)
    hard = O.pseudo_select(soft, 0.5, 0.2)
    _eq(ops.superpixel_expand(hard.to(dev), sup.to(dev), c), O.superpixel_expand(hard, sup, c), "expand ragged")
    rows = soft.permute(0, 2, 3, 1).reshape(b, -1, c).contiguous()
    for red in ("max", "sum", "mean"):
        got = ops.region_reduce(rows.to(dev), sup.reshape(b, -1).to(dev), red)
        want = O.region_reduce(rows, sup.reshape(b, -1, 1), red)
        if red == "max":
            _eq(got, want, "region max ragged")
        else:
            assert_close(got, want, rtol=1e-5, atol=1e-6, what="region " + red)
    got = ops.region_reduce(soft.to(dev), sup.to(dev), "max", planar=True)
    _eq(got, O.region_reduce(rows, sup.reshape(b, -1, 1), "max"), "region max planar")
    hot = O.index_onehot(hard, c).reshape(b, -1, c)
    _eq(ops.region_reduce(hot.to(dev), sup.reshape(b, -1).to(dev), "sum"), O.region_reduce(hot, sup.reshape(b, -1, 1), "sum"),
        "region sum i64")
    ent, _ = ops.entropy_uvem_weight(soft.to(dev))
    assert_close(ent, O.entropy(soft), rtol=RTOL, atol=1e-7, what="entropy ragged")
    s = 4
    lab = torch.randint(-1, c, (b, H, W), generator=g)
    _eq(ops.downscale_label(lab.to(dev), s, c, -1, 0.4), O.downscale_label(lab, s, c, -1, 0.4), "downscale ragged")
    h, w = max(H // s, 1), max(W // s, 1)
    k = 37
    feat = torch.randn(b, k, h, w, generator=g)
    protos = torch.randn(c, k, generator=g)
    flat = feat.permute(0, 2, 3, 1).reshape(-1, k)
    want = O.pearson_dist(flat, protos)
    assert_close(ops.pearson_dist_rows(flat.to(dev), protos.to(dev)), want, rtol=RTOL, atol=1e-6, what="pearson rows ragged")
    got = ops.pearson_dist_nchw(feat.to(dev), protos.to(dev)).permute(0, 2, 3, 1).reshape(-1, c)
    assert_close(got, want, rtol=RTOL, atol=1e-6, what="pearson nchw ragged")
    p1 = torch.randn(b, c, h, w, generator=g)
    refined = O.label_refine(sup, feat, p1, soft, protos, mode="all", temp=1.7)
    from uemda_b200 import mining
    got, _ = mining.refine_select(7, soft.to(dev), 1.7, feat=feat.to(dev), prototypes=protos.to(dev), pred1=p1.to(dev),
                                  sup=sup.to(dev))
    assert_close(got, refined, rtol=RTOL, atol=1e-7, what="refine ragged temp=1.7")
    lab_low = O.downscale_label(lab, s, c, -1, 0.4)
    sums, counts = ops.proto_accumulate(feat.to(dev), lab_low.to(dev), c)
    wsum, wcnt = O.class_feature_sums(feat, lab_low, c)
    assert_close(sums, wsum, rtol=RTOL, atol=1e-5, what="proto sums ragged")
    _eq(counts.float().reshape(c, 1), wcnt, "proto counts ragged")
    hist = ops.class_hist(lab.to(dev), c)
    whist, wvalid = O.class_histogram(lab, c)
    _eq(hist[:-1], whist, "class hist")
    assert int(hist[-1]) == int(wvalid)
    x = torch.rand(1000, generator=g) * 1.2 - 0.1
    _eq(ops.hist_f32(x.to(dev), 30, 0.0, 1.0), torch.histc(x, 30, 0.0, 1.0).long(), "histc")


@pytest.mark.parametrize("shape", [(2, 5, 72, 200, 9, 25), (1, 7, 40, 36, 20, 18), (3, 2, 33, 64, 3, 5), (1, 8, 64, 256, 4, 16),
                                   (2, 6, 50, 132, 50, 132), (1, 3, 1, 8, 1, 2)])
@pytest.mark.parametrize("temp", [2.0, 1.7])
def test_refine_column_kernel_shapes(dev, shape, temp):
    """Default configuration (all views, two heads, W % 4 == 0) at shapes that stress the column-walk kernel: partial
    and empty warps of the last 128-column strip, odd class counts, up-sampling ratios from 1 to 16, one-row maps."""
    from oracle import uem_oracle as O
    from uemda_b200 import mining
    b, c, H, W, h, w = shape
    g = torch.Generator().manual_seed(H * 1000 + W)
    soft = torch.softmax(torch.randn(b, c, H, W, generator=g) * 3, dim=1)
    sup = torch.randint(0, 11, (b, 1, H, W), generator=g)
    k = 19
    feat = torch.randn(b, k, h, w, generator=g)
    protos = torch.randn(c, k, generator=g)
    p1 = torch.randn(b, c, h, w, generator=g) * 4
    p2 = torch.randn(b, c, h, w, generator=g) * 4
    want = O.label_refine(sup, feat, [p1, p2], soft, protos, mode="all", temp=temp)
    got, _ = mining.refine_select(7, soft.to(dev), temp, feat=feat.to(dev), prototypes=protos.to(dev), pred1=p1.to(dev),
                                  pred2=p2.to(dev), sup=sup.to(dev))
    assert_close(got, want, rtol=RTOL, atol=1e-7, what="refine column kernel %s temp=%s" % (shape, temp))
    # per-(image, class) maxima that feed pseudo_selection come out of the same pass
    stats = got._uem_stats.stats
    hard = O.pseudo_select(got.cpu())
    from uemda_b200 import ops
    _eq(ops.pseudo_select_stats(got, stats, 0.8, 0.6, -1), hard, "selection from the kernel's own class statistics")


@pytest.mark.parametrize("shape", [(2, 5, 72, 200, 9, 25), (1, 7, 41, 37, 20, 18), (3, 2, 33, 64, 3, 5), (1, 8, 64, 256, 4, 16),
                                   (2, 6, 50, 131, 50, 131), (1, 3, 1, 8, 1, 2), (1, 1, 9, 9, 3, 3)])
@pytest.mark.parametrize("heads,temp", [(2, 1.0), (1, 1.0), (2, 1.7)])
def test_logits_pass_shapes(dev, shape, heads, temp):
    """a1-a4 at ragged shapes: odd widths, partial strips, one or two heads, temperature, up-sampling ratios 1..16."""
    from oracle import uem_oracle as O
    from uemda_b200 import ops
    b, c, H, W, h, w = shape
    g = torch.Generator().manual_seed(H * 977 + W)
    x1 = torch.randn(b, c, h, w, generator=g) * 4
    x2 = torch.randn(b, c, h, w, generator=g) * 4 if heads == 2 else None
    want = O.soft_from_logits(x1 / temp, None if x2 is None else x2 / temp, (H, W))
    out = ops.softmax_conf_entropy_argmax(x1.to(dev), None if x2 is None else x2.to(dev), size=(H, W), temp=temp)
    assert_close(out["soft"], want, rtol=RTOL, atol=1e-8, what="soft from logits %s" % (shape,))
    conf, arg = O.confidence_argmax(want)
    assert_close(out["conf"], conf, rtol=RTOL, atol=1e-8, what="conf")
    # entropy of the kernel's own probabilities: 1e-5.  Against the entropy of the reference's probabilities the term of a
    # dominant class (-p log p ~ 1 - p) moves by an ulp of p ~ 1, i.e. ~1e-7 absolute whatever the size of the entropy:
    # absolute tolerance 1e-6 there.
    assert_close(out["entropy"].reshape(-1), O.entropy(out["soft"].cpu()), rtol=RTOL, atol=1e-7, what="entropy of own soft")
    assert_close(out["entropy"].reshape(-1), O.entropy(want), rtol=RTOL, atol=1e-6, what="entropy from logits")
    if c > 1:
        top2 = want.topk(2, dim=1)[0]
        clear = (top2[:, 0] - top2[:, 1]) > 1e-5
        assert bool((out["argmax"].cpu()[clear] == arg[clear]).all())
    # argmax is exactly the first maximum of the kernel's own soft output (documented tie-break)
    _eq(out["argmax"], out["soft"].cpu().max(dim=1)[1], "argmax of own soft")
    only = ops.softmax_conf_entropy_argmax(x1.to(dev), None if x2 is None else x2.to(dev), size=(H, W), temp=temp, want=("argmax",))
    _eq(only["argmax"], out["argmax"], "argmax-only call")


def test_full_size_properties(dev):
    """BASELINE config 2 at full size (8x6x512x512, k=2048): size-independent properties instead of the
    (slow) oracle -- refined rows sum to ~1, hard labels equal the argmax wherever kept, thresholds
    respect cutoff_low, selection is idempotent under the cached and uncached class max, prototype
    update is linear in the features, and region max dominates every member pixel."""
    from uemda_b200 import mining, ops
    from uemda_b200.gast.alignment import Aligner
    from uemda_b200.gast.pseudo_generation import pseudo_selection
    from uemda_b200.synth import WORKLOADS, make_inputs
    wl = WORKLOADS["cfg2_isprs_8x6x512"]
    inp = make_inputs(wl, seed=11)
    d = _to(inp, dev)
    al = Aligner(_Log(), feat_channels=wl.k, class_num=wl.c, decay=0.996)
    al.prototypes = d["prototypes"].clone()
    refined, hard = mining.mine_step(al, d["sup"], d["feat"], [d["pred1"], d["pred2"]], d["soft"])
    s = refined.sum(dim=1)
    assert float((s - 1).abs().max()) < 1e-3  # sum/(sum+1e-7)
    assert float(refined.min()) >= 0 and float(refined.max()) <= 1
    kept = hard >= 0
    assert 0.05 < float(kept.float().mean()) < 0.999
    assert bool((hard[kept] == refined.argmax(dim=1)[kept]).all())
    conf = refined.max(dim=1)[0]
    assert float(conf[kept].min()) > 0.6
    _eq(pseudo_selection(refined, 0.8, 0.6, "tensor", -1), hard, "cached partials")
    _eq(pseudo_selection(refined.clone(), 0.8, 0.6, "tensor", -1), hard, "two-pass")
    # region max >= every member pixel, equality attained
    table = ops.region_reduce(d["soft"], d["sup"], "max", planar=True)
    ids = d["sup"].reshape(wl.b, -1, 1).expand(-1, -1, wl.c)
    gathered = torch.gather(table, 1, ids).reshape(wl.b, wl.H, wl.W, wl.c).permute(0, 3, 1, 2)
    assert bool((gathered >= d["soft"]).all())
    assert torch.equal(table, torch.zeros_like(table).scatter_reduce_(1, ids, d["soft"].permute(0, 2, 3, 1).reshape(wl.b, -1, wl.c),
                                                                     "amax", include_self=False))
    # prototype accumulation: linear in feat, counts are a checksum of the down-scaled labels
    down = al.downscale_gt(d["label_s"])
    s1, c1 = ops.proto_accumulate(d["feat_s"], down, wl.c)
    s2, _ = ops.proto_accumulate(d["feat_s"] * 2.0, down, wl.c)
    assert_close(s2, s1 * 2.0, rtol=1e-6, atol=1e-6, what="linearity")
    for ci in range(wl.c):
        assert int(c1[ci]) == int((down == ci).sum())
    ref_sum = torch.einsum("bkn,bcn->ck", d["feat_s"].reshape(wl.b, wl.k, -1).double(),
                           torch.nn.functional.one_hot(down.reshape(wl.b, -1) + 1, wl.c + 1)[..., 1:].permute(0, 2, 1).double())
    rms = ref_sum.pow(2).mean().sqrt().item()   # ~3e-6 of the rms is fp32 accumulation-order noise (see test_proto_sums_benchmarked_shapes)
    assert_close(s1, ref_sum.float(), rtol=RTOL, atol=1e-5 * rms, what="proto sums vs fp64")
    # expand is idempotent: expanding an already-expanded map changes nothing
    e1 = al.superpixel_expand(hard, d["sup"])
    _eq(al.superpixel_expand(e1, d["sup"]), e1, "expand idempotent")
    # determinism: the whole step is bit-reproducible run to run
    refined2, hard2 = mining.mine_step(al, d["sup"], d["feat"], [d["pred1"], d["pred2"]], d["soft"])
    assert torch.equal(refined, refined2) and torch.equal(hard, hard2)


def test_no_cpu_fallback(dev):
    from uemda_b200 import _lib, ops
    with pytest.raises(_lib.UemLibraryError):
        ops.class_max(torch.rand(1, 3, 8, 8))  # CPU tensor: must raise, never fall back


# ------------------------------------------------------------------------------------ workspace / chain housekeeping
def _small_inputs(dev, seed=11):
    from uemda_b200.synth import Workload, make_inputs
    wl = Workload("ws", 2, 6, 64, 96, 64, 16, 24)
    inp = make_inputs(wl, seed=seed)
    return wl, inp, _to(inp, dev)


def test_workspace_reuse_and_mixed_views(dev):
    """The fused chain keeps its workspace self-cleaning: a persistent workspace reused across calls, view subsets and
    the memset fallback path must give exactly what a fresh zeroed workspace gives."""
    from uemda_b200 import _lib, mining
    wl, inp, d = _small_inputs(dev)
    R = int(inp["ignore_id"]) + 1
    lib = _lib.load()
    ws = torch.zeros(lib.uem_mine_ws_bytes(wl.b, wl.c, wl.H, wl.W, wl.h, wl.w, wl.k, R), dtype=torch.uint8, device=dev)

    def run(views, ws_, **kw):
        return mining.refine_select(views, d["soft"], 2.0, feat=d["feat"], prototypes=d["prototypes"], pred1=d["pred1"],
                                    pred2=d["pred2"], sup=d["sup"], num_regions=R, select=(0.8, 0.6, -1), ws=ws_, **kw)

    fresh = {v: run(v, None) for v in (7, 4, 3, 6)}
    for v in (7, 7, 4, 3, 7, 6, 7):
        got = run(v, ws)
        _eq(got[0], fresh[v][0], "refined, views=%d on a reused workspace" % v)
        _eq(got[1], fresh[v][1], "hard, views=%d on a reused workspace" % v)
    # entropy / UVEM weight variant leaves the workspace just as clean
    a = run(7, ws, uvem=(0.2, 0.7, 4.0))
    b2 = run(7, ws, uvem=(0.2, 0.7, 4.0))
    for x, y in zip(a, b2):
        _eq(x, y, "repeat with uvem outputs")


def test_external_ignored_id_matches_internal(dev):
    """Multi-GPU form: the batch-global max id supplied by the caller (after an all-reduce) == computed in the chain."""
    from uemda_b200 import mining, ops
    wl, inp, d = _small_inputs(dev, seed=12)
    R = int(inp["ignore_id"]) + 1
    kw = dict(feat=d["feat"], prototypes=d["prototypes"], pred1=d["pred1"], pred2=d["pred2"], sup=d["sup"], num_regions=R,
              select=(0.8, 0.6, -1))
    ref = mining.refine_select(7, d["soft"], 2.0, **kw)
    ign = ops.i64_minmax(d["sup"])[1:].clone()
    got = mining.refine_select(7, d["soft"], 2.0, ignored_id=ign, **kw)
    _eq(got[0], ref[0], "refined with external ignored id")
    _eq(got[1], ref[1], "hard with external ignored id")
    # a different ignored id really changes which pixels the superpixel view skips
    other = torch.zeros_like(ign)
    diff = mining.refine_select(7, d["soft"], 2.0, ignored_id=other, **kw)
    assert not torch.equal(diff[0], ref[0])


def test_three_phase_miner_equals_update_prototype(dev):
    """ShardedMiner.local_stats -> exchange -> apply at world size 1 == Aligner.update_prototype."""
    from uemda_b200 import mining
    from uemda_b200.gast.alignment import Aligner, DownscaleLabel
    wl, inp, d = _small_inputs(dev, seed=13)

    def fresh():
        al = Aligner(_Log(), feat_channels=wl.k, class_num=wl.c, decay=0.996)
        al.downscale_gt = DownscaleLabel(wl.scale, wl.c, -1, 0.75)
        al.prototypes = d["prototypes"].clone()
        return al

    a = fresh()
    down_a = a.update_prototype(d["feat_s"], d["label_s"])
    b2 = fresh()
    miner = mining.ShardedMiner(b2)
    packed, down_b = miner.local_stats(d["sup"], d["feat_s"], d["label_s"])
    ignored = miner.apply(miner.exchange(packed), in_place=True)
    _eq(down_b, down_a, "down-scaled labels")
    _eq(b2.prototypes, a.prototypes, "prototypes after the three-phase update")
    assert int(ignored) == int(d["sup"].max())


def test_regeneration_driver_matches_oracle_per_tile(dev):
    """Next row (SURVEY 8f-1): offline regeneration = refine -> select -> uint8(label+1), reference batch size 1."""
    from oracle import uem_oracle as O
    from uemda_b200.regen import PseudoLabelRegenerator
    from uemda_b200.gast.alignment import Aligner
    from uemda_b200.synth import Workload, make_inputs
    wl = Workload("regen", 3, 6, 64, 64, 32, 16, 16)
    inp = make_inputs(wl, seed=21)
    # make tile 2 disagree on the max id so that the per-tile fallback is exercised too
    sup = inp["sup"].clone()
    sup[2][sup[2] == sup[2].max()] = int(sup[2].max()) + 3
    al = Aligner(_Log(), feat_channels=wl.k, class_num=wl.c)
    al.prototypes = inp["prototypes"].to(dev)
    want = []
    for i in range(wl.b):  # the reference walks the set with batch_size=1
        r = O.label_refine(sup[i:i + 1], inp["feat"][i:i + 1], [inp["pred1"][i:i + 1], inp["pred2"][i:i + 1]], inp["soft"][i:i + 1],
                           inp["prototypes"], mode="all", temp=2.0)
        want.append(O.pseudo_select(r, 0.8, 0.6, -1))
    want = (torch.cat(want) + 1).to(torch.uint8)
    batches = [{"soft": inp["soft"][:2].pin_memory(), "sup": sup[:2].pin_memory(), "feat": inp["feat"][:2].pin_memory(),
                "preds": [inp["pred1"][:2].pin_memory(), inp["pred2"][:2].pin_memory()], "names": ["t0", "t1"]},
               {"soft": inp["soft"][2:].pin_memory(), "sup": sup[2:].pin_memory(), "feat": inp["feat"][2:].pin_memory(),
                "preds": [inp["pred1"][2:].pin_memory(), inp["pred2"][2:].pin_memory()], "names": ["t2"]}]
    got = {}
    regen = PseudoLabelRegenerator(al, 0.8, 0.6, mode="all", temp=2.0, num_regions=int(sup.max()) + 1)
    n = regen.run(batches, lambda names, arr: got.update({nm: arr[j].copy() for j, nm in enumerate(names)}))
    assert n == 3 and sorted(got) == ["t0", "t1", "t2"]
    out = torch.from_numpy(np.stack([got["t0"], got["t1"], got["t2"]]))
    assert out.dtype == torch.uint8
    mism = int((out != want).sum())
    assert mism <= 2, "regenerated label mismatches vs oracle: %d" % mism
    # mixed batch (tiles 1 and 2 disagree on the ignored id) goes through the tile-by-tile path and agrees with the above
    mixed = regen.process(inp["soft"][1:].to(dev), sup[1:].to(dev), inp["feat"][1:].to(dev),
                          [inp["pred1"][1:].to(dev), inp["pred2"][1:].to(dev)])
    _eq(mixed, out[1:], "mixed-batch regeneration")
    # selection-only variant (pseudo_generation.py:138-151) is bit-exact
    plain = PseudoLabelRegenerator(None, 0.8, 0.6, refine=False).process(inp["soft"].to(dev))
    _eq(plain, (O.pseudo_select(inp["soft"], 0.8, 0.6, -1) + 1).to(torch.uint8), "selection-only regeneration")


def test_fused_fold_finalize_equals_two_step(dev):
    from uemda_b200 import ops
    wl, inp, d = _small_inputs(dev, seed=14)
    down = ops.downscale_label(d["label_s"], wl.scale, wl.c)
    sums, counts = ops.proto_accumulate(d["feat_s"], down, wl.c)
    _, want = ops.proto_finalize(sums, counts, d["prototypes"], decay=0.996, want_local=False)
    part = ops.proto_accumulate(d["feat_s"], down, wl.c, fold=False)
    got = ops.proto_fold_finalize(part, d["prototypes"], decay=0.996)
    _eq(got, want, "fused fold + finalize")
    state = d["prototypes"].clone()
    ops.proto_fold_finalize(part, state, decay=0.996, out=state)
    _eq(state, want, "in-place fused fold + finalize")


# ------------------------------------------------------------------------------------ next row 8f-2: PCL loss
def test_pcl_loss_golden_forward_backward(dev):
    """PrototypeContrastiveLoss forward + backward against the reference's own outputs (tests/golden/pcl_small.npz)."""
    import os
    from uemda_b200.loss import PrototypeContrastiveLoss
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "pcl_small.npz"))
    protos = torch.from_numpy(z["in_protos"]).to(dev)
    labels = torch.from_numpy(z["in_labels"]).to(dev)
    for temp in (8.0, 0.5):
        f = torch.from_numpy(z["in_feat"]).to(dev).requires_grad_(True)
        loss = PrototypeContrastiveLoss(temperature=temp, ignore_label=-1)(protos, f, labels)
        (loss * 1.0).backward()
        assert_close(loss.detach().reshape(1), torch.from_numpy(z["out_loss_t%g" % temp]).reshape(1), rtol=RTOL, atol=1e-7, what="pcl loss")
        assert_close(f.grad, torch.from_numpy(z["out_grad_t%g" % temp]), rtol=1e-4, atol=1e-7, what="pcl grad")


def test_pcl_loss_vs_oracle_config_shape(dev):
    """Config-2 feature shape (8,2048,32,32): loss and gradient vs the oracle's autograd; upstream gradient scaling;
    the (N,A) row form; all-ignored labels give NaN like the reference's mean over an empty set."""
    from oracle import uem_oracle as O
    from uemda_b200.loss import PrototypeContrastiveLoss
    g = torch.Generator().manual_seed(5)
    b, k, h, w, c = 8, 2048, 32, 32, 6
    protos = torch.randn(c, k, generator=g)
    lab = torch.randint(-1, c, (b, 1, h, w), generator=g)
    feat = torch.randn(b, k, h, w, generator=g) + 0.5 * protos[lab.clamp(min=0).squeeze(1)].permute(0, 3, 1, 2)
    f_ref = feat.clone().requires_grad_(True)
    want = O.pcl_loss(protos, f_ref, lab, temperature=8.0)
    (want * 0.5).backward()
    fn = PrototypeContrastiveLoss(temperature=8.0, ignore_label=-1)
    f = feat.to(dev).requires_grad_(True)
    loss = fn(protos.to(dev), f, lab.to(dev))
    (loss * 0.5).backward()
    assert_close(loss.detach().reshape(1), want.detach().reshape(1), rtol=RTOL, atol=1e-7, what="pcl loss cfg2")
    scale = float(f_ref.grad.abs().max())
    assert_close(f.grad, f_ref.grad, rtol=1e-4, atol=1e-5 * scale, what="pcl grad cfg2")
    # (N, A) rows
    rows = feat.permute(0, 2, 3, 1).reshape(-1, k)[:1000].contiguous()
    r_ref = rows.clone().requires_grad_(True)
    w2 = O.pcl_loss(protos, r_ref, lab.reshape(-1)[:1000], temperature=8.0)
    w2.backward()
    r = rows.to(dev).requires_grad_(True)
    l2 = fn(protos.to(dev), r, lab.reshape(-1)[:1000].to(dev))
    l2.backward()
    assert_close(l2.detach().reshape(1), w2.detach().reshape(1), rtol=RTOL, atol=1e-7, what="pcl loss rows")
    assert_close(r.grad, r_ref.grad, rtol=1e-4, atol=1e-5 * float(r_ref.grad.abs().max()), what="pcl grad rows")
    # nothing valid -> NaN (CrossEntropyLoss mean over zero elements)
    f3 = feat[:1].to(dev).requires_grad_(True)
    assert torch.isnan(fn(protos.to(dev), f3, torch.full((1, 1, h, w), -1, device=dev)))


def _grad_close(got, want, what):
    """gradients: 1e-5 relative to the largest entry of the map (entries are sums with cancellation: p_c - onehot_c)"""
    assert_close(got, want, rtol=RTOL, atol=RTOL * float(want.abs().max()), what=what)


def test_uvem_loss_golden_forward_backward(dev):
    """Next row 8f-3: fused up-sampling + UVEM/UPS cross-entropy, forward and backward, against the unmodified
    reference's loss_calc_uvem and its autograd gradients (tests/golden/uvem_loss_small.npz)."""
    import os
    import numpy as np
    from uemda_b200.gast.balance import ClassBalance, UPSLoss, UVEMLoss, loss_calc_uvem
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "uvem_loss_small.npz"))
    soft, label = torch.from_numpy(z["in_soft"]).to(dev), torch.from_numpy(z["in_label"]).to(dev)
    c = soft.shape[1]

    def run(tag, loss_fn, names, multi=True):
        xs = [torch.from_numpy(z[n]).to(dev).requires_grad_(True) for n in names]
        loss = loss_calc_uvem(xs if multi else xs[0], label, soft, loss_fn, multi=multi)
        loss.backward()
        assert_close(loss.detach().reshape(()), torch.from_numpy(z["out_%s_loss" % tag]), rtol=RTOL, atol=0, what=tag + " loss")
        for i, x in enumerate(xs):
            _grad_close(x.grad, torch.from_numpy(z["out_%s_grad%d" % (tag, i + 1)]), "%s grad head %d" % (tag, i + 1))

    run("uvem", UVEMLoss(m=0.2, threshold=0.7, gamma=4.0, class_num=c), ["in_x1", "in_x2"])
    run("uvem_single", UVEMLoss(m=0.2, threshold=0.7, gamma=4.0, class_num=c), ["in_x1"], multi=False)
    run("ups", UPSLoss(threshold=0.7, class_num=c), ["in_x1", "in_x2"])
    cb = ClassBalance(class_num=c, ignore_label=-1, decay=0.99, temperature=0.5)
    run("uvem_cb", UVEMLoss(m=0.2, threshold=0.7, gamma=4.0, class_balancer=cb, class_num=c), ["in_x1", "in_x2"])
    assert_close(cb.freq, torch.from_numpy(z["out_uvem_cb_freq"]), rtol=RTOL, atol=1e-8, what="class frequency after two heads")


@pytest.mark.parametrize("shape", [(2, 6, 32, 32, 512, 512), (1, 7, 5, 7, 33, 50), (2, 3, 4, 4, 4, 4), (1, 5, 9, 3, 20, 64),
                                   (1, 2, 1, 1, 8, 8), (1, 8, 6, 10, 96, 160)])
def test_uvem_loss_vs_oracle_shapes(dev, shape):
    """Fused loss at the config-2 shape and at ragged ones (non-integer ratios, no up-sampling, a 1x1 head, odd class
    counts) against the oracle's autograd; the gradient kernel is a gather, so two runs are bit-identical."""
    from oracle import uem_oracle as O
    from uemda_b200.gast.balance import UVEMLoss, loss_calc_uvem
    b, c, h, w, H, W = shape
    g = torch.Generator().manual_seed(h * 131 + W)
    x1 = torch.randn(b, c, h, w, generator=g) * 2
    x2 = torch.randn(b, c, h, w, generator=g) * 2
    soft = torch.softmax(torch.randn(b, c, H, W, generator=g) * 3, dim=1)
    # get_weight has unbounded slope where the entropy meets the threshold (w = x^(1/gamma), x -> 0): an entropy that
    # differs in its last bit moves the weight by ~1e-3 there (same caveat as test_oracle_mining_step).  That is the
    # conditioning of the reference's formula, not of the fused kernels: keep the test pixels 2e-3 away from it.
    u = O.entropy(soft).reshape(b, 1, H, W)
    peaked = torch.full((c,), 1e-3)
    peaked[0] = 1.0 - 1e-3 * (c - 1)
    soft = torch.where((u - 0.7).abs() < 2e-3, peaked.view(1, c, 1, 1), soft)
    label = torch.randint(-1, c, (b, H, W), generator=g)
    cx = [x.clone().requires_grad_(True) for x in (x1, x2)]
    want, _ = O.uvem_loss_calc(cx, label, soft, m=0.2, threshold=0.7, gamma=4.0)
    want.backward()
    fn = UVEMLoss(m=0.2, threshold=0.7, gamma=4.0, class_num=c)
    gx = [x.to(dev).requires_grad_(True) for x in (x1, x2)]
    if (h, w) == (H, W):   # loss_calc_uvem only fuses when it has to up-sample: call the fused form directly
        loss = fn.fused_heads(gx, label.to(dev), soft.to(dev)) / 2
    else:
        loss = loss_calc_uvem(gx, label.to(dev), soft.to(dev), fn)
    loss.backward()
    assert_close(loss.detach().reshape(()), want.detach(), rtol=RTOL, atol=0, what="fused loss %s" % (shape,))
    for i in range(2):
        _grad_close(gx[i].grad, cx[i].grad, "fused grad head %d %s" % (i + 1, shape))
    again = [x.to(dev).requires_grad_(True) for x in (x1, x2)]
    (fn.fused_heads(again, label.to(dev), soft.to(dev)) / 2).backward()
    for i in range(2):
        _eq(again[i].grad, gx[i].grad.cpu(), "gradient is deterministic")
    # the unfused drop-in path (PyTorch cross-entropy on up-sampled logits) agrees
    import torch.nn.functional as tnf
    ux = [x.to(dev).requires_grad_(True) for x in (x1, x2)]
    up = [tnf.interpolate(x, size=(H, W), mode="bilinear", align_corners=True) for x in ux]
    unfused = (fn(up[0], label.to(dev), soft.to(dev)) + fn(up[1], label.to(dev), soft.to(dev))) / 2
    assert_close(unfused.detach().reshape(()), loss.detach().reshape(()), rtol=RTOL, atol=0, what="fused vs unfused loss")


def test_exchange_pack_and_fold_kernels(dev):
    """8e: the one-launch pack / rank-ordered fold of the exchange vector equal the elementwise torch form bit for bit."""
    from uemda_b200 import mining, ops
    g = torch.Generator().manual_seed(5)
    c, k, world = 6, 2048, 3
    rows = []
    for r in range(world):
        sums = torch.randn(c, k, generator=g) * 1000
        counts = torch.randint(0, 1 << 40, (c,), generator=g)
        mx = torch.randint(0, 1 << 33, (1,), generator=g)
        want = mining.pack_local(sums, counts, mx)                       # CPU tensors: elementwise torch form
        got = ops.pack_local(sums.to(dev), counts.to(dev), mx.to(dev))
        _eq(got, want, "pack rank %d" % r)
        rows.append(want)
    gathered = torch.stack(rows)
    ws, wc, wm = mining.fold_gathered(gathered, c, k)                    # CPU form
    gs, gc, gm = ops.fold_gathered(gathered.to(dev), c, k)
    _eq(gs, ws, "folded sums")
    _eq(gc, wc, "folded counts")
    _eq(gm, wm, "folded max id")


def test_staged_region_phase_equals_fused_chain(dev):
    """8e: region half of the chain run on its own (one step ahead of the exchange) + refine/select with
    UEM_VIEW_REGIONS_READY give bit-identical results to the single fused call, leave the workspace clean (second
    round on the same workspace), and expose the rank-local max superpixel id."""
    from uemda_b200 import mining
    from uemda_b200.synth import WORKLOADS, make_inputs
    wl = WORKLOADS["tiny"]
    for seed in (3, 4):
        inp = _to(make_inputs(wl, seed=seed), dev)
        R = int(inp["ignore_id"]) + 1
        kw = dict(feat=inp["feat"], prototypes=inp["prototypes"], pred1=inp["pred1"], pred2=inp["pred2"], sup=inp["sup"],
                  num_regions=R, select=(0.8, 0.6, -1), uvem=(0.2, 0.7, 4.0))
        want = mining.refine_select(7, inp["soft"], 2.0, **kw)
        if seed == 3:
            ws = mining.mine_workspace(inp["soft"], R, wl.h, wl.w, wl.k)
        local = mining.region_phase(inp["soft"], inp["sup"], 2.0, R, ws, wl.h, wl.w, wl.k)
        assert int(local.item()) == int(inp["sup"].max().item())
        ignored = local.clone()   # a single rank: the global id is the local one
        got = mining.refine_select(7, inp["soft"], 2.0, ignored_id=ignored, ws=ws, regions_ready=True, **kw)
        for a, b2, name in zip(got, want, ("refined", "hard", "entropy", "uvem weight")):
            _eq(a, b2, "staged " + name)
        assert int(local.item()) == 0, "the selection kernel zeroes the max-id slot again"


@pytest.mark.parametrize("world", [1, 2, 3])
def test_region_phase_carries_the_id_send(dev, world):
    """8e: the id part of a step's exchange issued by the LAST CTA of the region-max kernel (uem_mine_region_phase_xchg_f32)
    instead of a launch of its own.  ``world`` ranks emulated on one device, launches issued in an order in which nothing
    ever has to wait (only the last rank polls: every other id is already there).  Every rank has a different max
    superpixel id; 5 steps > depth exercise slot reuse and the acknowledgements; the staged chain fed with the exchanged
    id equals the one-call chain given the same batch-global id."""
    from uemda_b200 import mining, ops
    from uemda_b200.exchange import PeerExchange
    from uemda_b200.synth import WORKLOADS, make_inputs
    wl = WORKLOADS["tiny"]
    c, k, depth = wl.c, wl.k, 3
    xs = PeerExchange.local_only(world, c, k, depth=depth, device=dev)
    inps = [_to(make_inputs(wl, seed=20 + r), dev) for r in range(world)]
    R = max(int(i["ignore_id"]) for i in inps) + 1 + world
    for r, inp in enumerate(inps):   # rank r's largest id is R - 1 - r: the ranks disagree about the max
        inp["sup"] = torch.where(inp["sup"] == int(inp["ignore_id"]), torch.full_like(inp["sup"], R - 1 - r), inp["sup"])
    wss = [mining.mine_workspace(inps[r]["soft"], R, wl.h, wl.w, wl.k) for r in range(world)]
    banks = [inps[0]["prototypes"].clone() for _ in range(world)]
    gids = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
    for step in range(5):
        slot = step % depth
        locals_ = []
        for r in range(world):
            last = r == world - 1
            loc = mining.region_phase(inps[r]["soft"], inps[r]["sup"], 2.0, R, wss[r], wl.h, wl.w, wl.k,
                                      exchange=(xs[r], slot, gids[r] if last else None))
            locals_.append(int(loc.item()))
        assert locals_ == [R - 1 - r for r in range(world)]
        assert int(gids[world - 1]) == R - 1, "batch-global id polled by the region-max kernel's tail"
        for r in range(world - 1):
            xs[r].wait_max_id(slot, out=gids[r])
            assert int(gids[r]) == R - 1
        # the sums of the step follow with the same sequence number, then the fold acknowledges the slot
        parts = [ops.proto_accumulate(inps[r]["feat_s"], mining_down(inps[r], wl), c, -1, fold=False) for r in range(world)]
        for r in range(world):
            xs[r].send(parts[r], None, slot, part="sums")
        for r in range(world):
            xs[r].fold_finalize(slot, banks[r], eps=1e-7, decay=0.9, out=banks[r])
            assert xs[r].status() == 0
            assert torch.equal(banks[r], banks[0])
        # refine + selection of every rank on the staged regions with the exchanged id == the one-call chain given that id
        for r in range(world):
            inp = inps[r]
            kw = dict(feat=inp["feat"], prototypes=inp["prototypes"], pred1=inp["pred1"], pred2=inp["pred2"], sup=inp["sup"],
                      num_regions=R, select=(0.8, 0.6, -1), uvem=(0.2, 0.7, 4.0))
            got = mining.refine_select(7, inp["soft"], 2.0, ignored_id=gids[r], ws=wss[r], regions_ready=True, **kw)
            want = mining.refine_select(7, inp["soft"], 2.0, ignored_id=gids[r].clone(), **kw)
            for a, b2, name in zip(got, want, ("refined", "hard", "entropy", "uvem weight")):
                _eq(a, b2, "rank %d staged %s" % (r, name))


def test_refused_region_phase_sends_nothing_later(dev):
    """8e: an id-carrying region phase that is refused (a region capacity past the shared-memory table) sends nothing,
    and a plain region phase issued next on the same thread does not carry that send either: the exchange region stays
    untouched and no poll times out."""
    from uemda_b200 import mining
    from uemda_b200.exchange import PeerExchange
    from uemda_b200.synth import WORKLOADS, make_inputs
    wl = WORKLOADS["tiny"]
    (peer,) = PeerExchange.local_only(1, wl.c, wl.k, device=dev)
    inp = _to(make_inputs(wl, seed=7), dev)
    gid = torch.zeros(1, dtype=torch.int64, device=dev)
    big = 20000
    ws_big = mining.mine_workspace(inp["soft"], big, wl.h, wl.w, wl.k)
    with pytest.raises(RuntimeError):
        mining.region_phase(inp["soft"], inp["sup"], 2.0, big, ws_big, wl.h, wl.w, wl.k, exchange=(peer, 0, gid))
    R = int(inp["ignore_id"]) + 1
    ws = mining.mine_workspace(inp["soft"], R, wl.h, wl.w, wl.k)
    local = mining.region_phase(inp["soft"], inp["sup"], 2.0, R, ws, wl.h, wl.w, wl.k)
    assert int(local.item()) == int(inp["sup"].max().item())
    region = peer._keep[peer.rank]
    assert int(region.count_nonzero()) == 0, "the exchange region was written by a call that asked for no exchange"
    assert int(gid.item()) == 0
    assert peer.status() == 0


def mining_down(inp, wl):
    from uemda_b200.gast.alignment import DownscaleLabel
    return DownscaleLabel(wl.scale, wl.c, -1, 0.75)(inp["label_s"])


def test_pack_from_partials_equals_fold_then_pack(dev):
    """8e: folding the per-image prototype partials and packing them in ONE launch is bit-identical to fold -> pack."""
    from uemda_b200 import ops
    g = torch.Generator().manual_seed(11)
    b, c, k, h, w = 5, 6, 96, 8, 12
    feat = torch.randn(b, k, h, w, generator=g).to(dev)
    lab = torch.randint(-1, c, (b, 1, h, w), generator=g).to(dev)
    mx = torch.tensor([1234567], dtype=torch.int64, device=dev)
    sums, counts = ops.proto_accumulate(feat, lab, c, -1)
    want = ops.pack_local(sums, counts, mx)
    got = ops.pack_local_partials(ops.proto_accumulate(feat, lab, c, -1, fold=False), mx)
    _eq(got, want, "pack from partials")
    out = (torch.empty((c, k), device=dev), torch.empty(c, dtype=torch.int64, device=dev), torch.empty(1, dtype=torch.int64, device=dev))
    s2, c2, m2 = ops.fold_gathered(torch.stack([want, want]), c, k, out=out)
    assert s2.data_ptr() == out[0].data_ptr()
    _eq(c2, counts * 2, "folded counts into static buffers")
    _eq(m2, mx, "folded max id into static buffers")


@pytest.mark.parametrize("regions,uniform_image", [(9001, False), (20000, False), (300, True)])
def test_chain_region_capacity_paths(dev, regions, uniform_image):
    """Region tables that do NOT fit shared memory (config 5's 16k regions take the global-table path with per-call
    zeroing instead of the self-cleaning one), sparse ids, and an image that consists of the ignored id only."""
    from oracle import uem_oracle as O
    from uemda_b200 import mining
    g = torch.Generator().manual_seed(regions)
    b, c, H, W, h, w, k = 2, 6, 96, 128, 6, 8, 24
    soft = torch.softmax(torch.randn(b, c, H, W, generator=g) * 2, dim=1)
    sup = torch.randint(0, regions, (b, 1, H // 4, W // 4), generator=g).repeat_interleave(4, 2).repeat_interleave(4, 3)
    sup[0, 0, :3, :] = regions - 1                       # make sure the batch max (the ignored id) is present
    if uniform_image:
        sup[1] = regions - 1                             # image 1: every pixel carries the ignored id
    feat = torch.randn(b, k, h, w, generator=g)
    protos = torch.randn(c, k, generator=g)
    p1 = torch.randn(b, c, h, w, generator=g) * 2
    p2 = torch.randn(b, c, h, w, generator=g) * 2
    want = O.label_refine(sup, feat, [p1, p2], soft, protos, mode="all", temp=2.0)
    want_hard = O.pseudo_select(want)
    kw = dict(feat=feat.to(dev), prototypes=protos.to(dev), pred1=p1.to(dev), pred2=p2.to(dev), sup=sup.to(dev),
              select=(0.8, 0.6, -1))
    for nr in (None, regions):
        got, hard = mining.refine_select(7, soft.to(dev), 2.0, num_regions=nr, **kw)
        assert_close(got, want, rtol=RTOL, atol=1e-7, what="refined, %d regions (capacity %s)" % (regions, nr))
        mism = int((hard.cpu() != want_hard).sum())
        assert mism <= 2, "label mismatches %d" % mism
    # same workspace twice (the non-self-cleaning path must leave it clean as well)
    ws = mining.mine_workspace(soft.to(dev), regions, h, w, k)
    a = mining.refine_select(7, soft.to(dev), 2.0, num_regions=regions, ws=ws, **kw)
    b2 = mining.refine_select(7, soft.to(dev), 2.0, num_regions=regions, ws=ws, **kw)
    _eq(a[0], b2[0], "workspace reuse, refined")
    _eq(a[1], b2[1], "workspace reuse, hard")


# ------------------------------------------------------------------------------------ round-2 regressions (ADVICE r1)
@pytest.mark.parametrize("mode", ["all", "s", "p", "l"])
@pytest.mark.parametrize("num_regions", [None, "tight", 7000])
def test_label_refine_then_selection_every_mode(golden, dev, mode, num_regions):
    """label_refine(mode) -> pseudo_selection must equal pseudo_selection of a plain copy of the refined map (which takes
    the two-pass class-max path) for every view subset and for region capacities on both sides of the shared-memory
    table limit: the class statistics handed from the refine call to the selection must be those of THIS call on the
    non-self-cleaning paths too ('p' / 'l' have no superpixel view; R = 7000 exceeds the table)."""
    from uemda_b200.gast.pseudo_generation import pseudo_selection
    g = golden
    al = _aligner(g, dev)
    if num_regions == "tight":
        al.num_regions = g.ignore_id + 1
    elif num_regions is not None:
        al.num_regions = num_regions
    preds = [p.to(dev) for p in g.preds()] if g.two_heads else g.preds().to(dev)
    for _ in range(2):   # twice: the second call runs on whatever the first left behind
        refined = al.label_refine(g.t("in_sup", dev), g.t("in_feat", dev), preds, g.t("in_soft", dev), mode=mode, temp=2.0)
        assert_close(refined, g.t("out_refine_" + mode), rtol=RTOL, atol=1e-7, what="label_refine " + mode)
        cached = pseudo_selection(refined, 0.8, 0.6, "tensor", -1)
        plain = pseudo_selection(refined.clone(), 0.8, 0.6, "tensor", -1)
        _eq(cached, plain, "selection with cached class statistics, mode %s, R %s" % (mode, num_regions))
        assert int((plain != -1).sum()) > 0


def test_stats_cache_is_not_trusted_blindly(golden, dev):
    """The side-channel cache must not be used for a tensor it does not describe (in-place edit, other class count)."""
    from uemda_b200.gast.pseudo_generation import pseudo_selection
    g = golden
    al = _aligner(g, dev)
    preds = [p.to(dev) for p in g.preds()] if g.two_heads else g.preds().to(dev)
    refined = al.label_refine(g.t("in_sup", dev), g.t("in_feat", dev), preds, g.t("in_soft", dev), mode="all", temp=2.0)
    cache = refined._uem_stats
    assert cache.valid_for(refined)
    other = refined[:, : g.c - 1].contiguous()
    other._uem_stats = cache                      # wrong class count
    assert not cache.valid_for(other)
    _eq(pseudo_selection(other, 0.8, 0.6, "tensor", -1), pseudo_selection(other.clone(), 0.8, 0.6, "tensor", -1), "foreign cache")
    refined.mul_(0.5)                             # in-place edit bumps the version
    assert not cache.valid_for(refined)
    _eq(pseudo_selection(refined, 0.8, 0.6, "tensor", -1), pseudo_selection(refined.clone(), 0.8, 0.6, "tensor", -1), "stale cache")


def test_out_of_range_ids_raise_under_strict_asserts(golden, dev):
    """Superpixel ids outside [0, num_regions): the reference's scatter/gather raises; so does the drop-in under
    strict_asserts (status word of the workspace read back and cleared)."""
    from uemda_b200 import config
    g = golden
    al = _aligner(g, dev)
    al.num_regions = 5   # far too small
    preds = [p.to(dev) for p in g.preds()] if g.two_heads else g.preds().to(dev)
    assert config.strict_asserts
    with pytest.raises(RuntimeError):
        al.label_refine(g.t("in_sup", dev), g.t("in_feat", dev), preds, g.t("in_soft", dev), mode="all", temp=2.0)
    with pytest.raises(RuntimeError):
        al.superpixel_expand(g.t("out_select_soft", dev), g.t("in_sup", dev))
    neg = g.t("in_sup", dev).clone()
    neg[0, 0, 0, 0] = -3
    al.num_regions = None
    with pytest.raises(RuntimeError):
        al.label_refine(neg, g.t("in_feat", dev), preds, g.t("in_soft", dev), mode="s", temp=2.0)
    al.num_regions = g.ignore_id + 1   # and a good call afterwards is clean
    got = al.label_refine(g.t("in_sup", dev), g.t("in_feat", dev), preds, g.t("in_soft", dev), mode="all", temp=2.0)
    assert_close(got, g.t("out_refine_all"), rtol=RTOL, atol=1e-7, what="label_refine after a rejected call")


@pytest.mark.parametrize("hw", [(33, 33), (5, 7), (17, 2)])
def test_pcl_loss_odd_feature_maps(dev, hw):
    """4-D feature maps whose h*w is not a multiple of 4 (33x33, 65x65 decoders): the reference accepts any shape."""
    from oracle import uem_oracle as O
    from uemda_b200.loss import PrototypeContrastiveLoss
    h, w = hw
    g = torch.Generator().manual_seed(h * 100 + w)
    b, k, c = 3, 64, 5
    protos = torch.randn(c, k, generator=g)
    lab = torch.randint(-1, c, (b, 1, h, w), generator=g)
    feat = torch.randn(b, k, h, w, generator=g)
    f_ref = feat.clone().requires_grad_(True)
    want = O.pcl_loss(protos, f_ref, lab, temperature=8.0)
    want.backward()
    f = feat.to(dev).requires_grad_(True)
    loss = PrototypeContrastiveLoss(8.0, -1)(protos.to(dev), f, lab.to(dev))
    loss.backward()
    assert_close(loss.detach().reshape(1), want.detach().reshape(1), rtol=RTOL, atol=1e-7, what="pcl loss odd map")
    assert_close(f.grad, f_ref.grad, rtol=1e-4, atol=1e-5 * float(f_ref.grad.abs().max()), what="pcl grad odd map")


def test_regeneration_run_reuses_buffers_and_streams(dev):
    """PseudoLabelRegenerator.run over many small batches (double-buffered staging + two reused pinned output buffers):
    every batch's output must equal process() of the same batch run on its own."""
    from uemda_b200.gast.alignment import Aligner
    from uemda_b200.regen import PseudoLabelRegenerator
    from uemda_b200.synth import Workload, make_inputs
    wl = Workload("regen2", 2, 6, 64, 64, 32, 16, 16)
    batches = []
    for i in range(7):
        inp = make_inputs(wl, seed=100 + i, with_source=False)
        batches.append({"soft": inp["soft"].pin_memory(), "sup": inp["sup"].pin_memory(), "feat": inp["feat"].pin_memory(),
                        "preds": [inp["pred1"].pin_memory(), inp["pred2"].pin_memory()], "names": ["b%d_%d" % (i, j) for j in range(2)]})
    al = Aligner(_Log(), feat_channels=wl.k, class_num=wl.c, decay=0.996)
    al.prototypes = inp["prototypes"].to(dev)
    regen = PseudoLabelRegenerator(al, 0.8, 0.6, mode="all", temp=2.0, num_regions=int(inp["ignore_id"]) + 1)
    got = {}
    n = regen.run(batches, lambda names, arr: got.update({nm: arr[j].copy() for j, nm in enumerate(names)}))
    assert n == 14 and len(got) == 14
    for i, bt in enumerate(batches):
        want = regen.process(bt["soft"].to(dev), bt["sup"].to(dev), bt["feat"].to(dev), [p.to(dev) for p in bt["preds"]]).cpu().numpy()
        for j in range(2):
            assert (got["b%d_%d" % (i, j)] == want[j]).all(), "batch %d tile %d" % (i, j)


# ------------------------------------------------------------------------------------ benchmarked shapes (VERDICT r1 item 1)
def _feat_set(kind, b, k, h, w, c, seed):
    """SURVEY 8(d) feature sets: 'generic' = N(0,1) + 0.5 proto[class], instance-normalised; 'near' = the cancellation
    edge case, proto[class] + 0.05 noise (Pearson r -> 1, dist ~ 5e-4)."""
    g = torch.Generator().manual_seed(seed)
    protos = torch.randn(c, k, generator=g)
    cls = torch.randint(0, c, (b, h, w), generator=g)
    if kind == "near":
        feat = protos[cls].permute(0, 3, 1, 2) + 0.05 * torch.randn(b, k, h, w, generator=g)
    else:
        feat = torch.randn(b, k, h, w, generator=g) + 0.5 * protos[cls].permute(0, 3, 1, 2)
        feat = (feat - feat.mean(dim=(2, 3), keepdim=True)) / (feat.std(dim=(2, 3), keepdim=True) + 1e-5)
    return feat.contiguous(), protos, cls


@pytest.mark.parametrize("b,c,h,w", [(8, 6, 32, 32), (2, 7, 64, 64), (6, 7, 64, 64), (3, 6, 32, 32)])
@pytest.mark.parametrize("kind", ["generic", "near"])
def test_pearson_benchmarked_shapes(dev, b, c, h, w, kind):
    """Pearson distance at the BENCHMARKED feature shapes, k = 2048: config 2 (8 x 32x32: the TMA kernel splits k over 4
    CTAs per pixel tile), config 3's 64x64 maps at k-splits 4 and 1, and a batch that takes the 8-way split; on the
    generic and on the near-prototype (cancellation) feature sets.  Contract (SURVEY section 7): abs 1e-6 on dist, and
    1e-5 relative wherever dist is not a cancellation result; the measured error is printed."""
    from oracle import uem_oracle as O
    from uemda_b200 import ops
    k = 2048
    feat, protos, _ = _feat_set(kind, b, k, h, w, c, seed=b * 100 + h)
    rows = feat.permute(0, 2, 3, 1).reshape(-1, k)
    want = O.pearson_dist(rows, protos)                                   # the reference's fp32 centre-then-dot form
    want64 = O.pearson_dist(rows.double(), protos.double())
    got = ops.pearson_dist_nchw(feat.to(dev), protos.to(dev))
    got_rows = got.permute(0, 2, 3, 1).reshape(-1, c).cpu()
    err = (got_rows - want).abs().max().item()
    err64 = (got_rows.double() - want64).abs().max().item()
    ref64 = (want.double() - want64).abs().max().item()
    print("pearson %s b=%d hw=%d: min dist %.3e, |ours-ref32| %.2e, |ours-fp64| %.2e, |ref32-fp64| %.2e"
          % (kind, b, h * w, want64.min().item(), err, err64, ref64))
    assert_close(got_rows, want, rtol=RTOL, atol=1e-6, what="pearson nchw k=2048 %s" % kind)
    assert err64 <= max(4 * ref64, 5e-7), "one-pass sums lose accuracy vs fp64: %.2e (reference %.2e)" % (err64, ref64)
    rws = ops.pearson_dist_rows(rows[:4096].contiguous().to(dev), protos.to(dev)).cpu()
    assert_close(rws, want[:4096], rtol=RTOL, atol=1e-6, what="pearson rows k=2048 %s" % kind)
    # 1/dist (what label_refine consumes, alignment.py:216): same tolerance on the reciprocal of a well-conditioned dist
    if kind == "generic":
        rec = ops.pearson_dist_nchw(feat.to(dev), protos.to(dev), reciprocal=True).permute(0, 2, 3, 1).reshape(-1, c).cpu()
        assert_close(rec, 1.0 / want, rtol=RTOL, atol=1e-6, what="1/pearson k=2048")


@pytest.mark.parametrize("b,c,h,w", [(8, 6, 32, 32), (2, 7, 64, 64), (16, 7, 64, 64)])
def test_proto_sums_benchmarked_shapes(dev, b, c, h, w):
    """Masked prototype sums + EMA at the benchmarked feature shapes (k = 2048) against the oracle's fp32 sums and fp64.
    Entries are sums of ~b*h*w/c signed terms: fp32 accumulation-order noise is ~3e-6 of the rms of the sums (the oracle's
    own fp32 sums sit that far from fp64), hence atol = 1e-5 x rms next to rtol 1e-5; local means and the EMA-updated
    prototypes (what north_star names) are held to 1e-5 relative with atol 1e-7 / 1e-6."""
    from oracle import uem_oracle as O
    from uemda_b200 import ops
    k = 2048
    feat, protos, cls = _feat_set("generic", b, k, h, w, c, seed=7 + b)
    g = torch.Generator().manual_seed(3)
    lab = torch.where(torch.rand(b, h, w, generator=g) < 0.1, torch.full_like(cls, -1), cls).unsqueeze(1)
    want, wcnt = O.class_feature_sums(feat, lab, c)
    onehot = torch.nn.functional.one_hot(lab.reshape(b, -1) + 1, c + 1)[..., 1:].permute(0, 2, 1).double()
    want64 = torch.einsum("bkn,bcn->ck", feat.reshape(b, k, -1).double(), onehot)
    sums, counts = ops.proto_accumulate(feat.to(dev), lab.to(dev), c)
    _eq(counts.float().reshape(c, 1), wcnt, "counts")
    rms = want64.pow(2).mean().sqrt().item()
    e32 = (sums.cpu() - want).abs().max().item()
    e64 = (sums.cpu().double() - want64).abs().max().item()
    r64 = (want.double() - want64).abs().max().item()
    print("proto sums b=%d hw=%d: rms %.1f, |ours-ref32| %.2e, |ours-fp64| %.2e, |ref32-fp64| %.2e" % (b, h * w, rms, e32, e64, r64))
    assert_close(sums, want, rtol=RTOL, atol=1e-5 * rms, what="proto sums k=2048")
    assert e64 <= max(4 * r64, 1e-5 * rms)
    wl, _ = O.local_prototypes(feat, lab, protos, c)
    local, new = ops.proto_finalize(sums, counts, protos.to(dev), decay=0.996)
    assert_close(local, wl, rtol=RTOL, atol=1e-7, what="local prototypes k=2048")
    assert_close(new, O.ema(protos, wl, 0.996), rtol=RTOL, atol=1e-6, what="EMA prototypes k=2048")


# ------------------------------------------------------------------------------------ device-side exchange (SURVEY 8e)
@pytest.mark.parametrize("world,depth", [(4, 3), (2, 2), (1, 3), (8, 3)])
def test_peer_exchange_emulated_ranks(dev, world, depth):
    """uem_xchg_send / wait_maxid / fold_finalize with `world` emulated ranks whose symmetric regions all live on this GPU
    (every launch is issued in an order in which its flags are already set, so nothing ever spins: one GPU must not run
    kernels that wait for each other).  7 steps > depth exercise slot reuse and the acknowledgement protocol.  Checked
    against the NCCL form's arithmetic (pack -> rank-ordered fold -> EMA), a one-rank run over the concatenated batch,
    and for bit-identical banks across ranks."""
    from uemda_b200 import ops
    from uemda_b200.exchange import PeerExchange
    c, k, h, w, b = 6, 256, 8, 8, 2
    g = torch.Generator().manual_seed(world * 10 + depth)
    xs = PeerExchange.local_only(world, c, k, depth=depth, device=dev)
    protos0 = torch.randn(c, k, generator=g).to(dev)
    banks = [protos0.clone() for _ in range(world)]
    bank_nccl = protos0.clone()
    bank_one = protos0.clone()
    for step in range(7):
        slot = step % depth
        feats = [torch.randn(b, k, h, w, generator=g).to(dev) for _ in range(world)]
        labs = [torch.randint(-1, c if step != 3 else 2, (b, 1, h, w), generator=g).to(dev) for _ in range(world)]   # step 3: empty classes
        ids = [torch.randint(0, 1 << 40, (1,), generator=g).to(dev) for _ in range(world)]
        hists = [ops.class_hist(labs[r], c) for r in range(world)]
        parts = [ops.proto_accumulate(feats[r], labs[r], c, -1, fold=False) for r in range(world)]
        gid = torch.zeros(1, dtype=torch.int64, device=dev)
        if step % 2 == 0:   # one launch per rank; the last sender finds every other id already there and may poll for the global id
            for r in range(world):
                xs[r].send(parts[r], ids[r], slot, hist=hists[r], global_id_out=gid if r == world - 1 else None)
        else:               # the split form: ids early (right after the region pass), sums later; same sequence number
            for r in range(world):
                xs[r].send(None, ids[r], slot, global_id_out=gid if r == world - 1 else None, part="id")
            for r in range(world):
                xs[r].send(parts[r], None, slot, hist=hists[r], part="sums")
        assert int(gid) == max(int(i) for i in ids), "global id from the fused send"
        got_ids, got_hist = [], []
        for r in range(world):
            got_ids.append(xs[r].wait_max_id(slot))
            new, sums, counts, hist = xs[r].fold_finalize(slot, banks[r], eps=1e-7, decay=0.9, out=banks[r], want_sums=True, want_hist=True)
            got_hist.append(hist)
            if r == 0:
                sums0, counts0 = sums, counts
        for r in range(world):
            assert xs[r].status() == 0
            assert int(got_ids[r]) == max(int(i) for i in ids)
            _eq(got_hist[r], torch.stack(hists).sum(0), "global class histogram")
            assert torch.equal(banks[r], banks[0]), "prototype bank differs across ranks at step %d" % step
        # NCCL form: fp64 pack -> rank-ordered fold -> EMA
        gathered = torch.stack([ops.pack_local_partials(parts[r], ids[r]) for r in range(world)])
        s2, n2, m2 = ops.fold_gathered(gathered, c, k)
        _eq(counts0, n2, "counts vs the all-gather form")
        assert_close(sums0, s2, rtol=1e-6, atol=1e-5, what="sums vs the all-gather form")
        _, bank_nccl = ops.proto_finalize(s2, n2, bank_nccl, decay=0.9, want_local=False)
        assert_close(banks[0], bank_nccl, rtol=1e-5, atol=1e-6, what="bank vs the all-gather form")
        # one rank over the concatenated batch
        s1, n1 = ops.proto_accumulate(torch.cat(feats), torch.cat(labs), c, -1)
        _, bank_one = ops.proto_finalize(s1, n1, bank_one, decay=0.9, want_local=False)
        assert_close(banks[0], bank_one, rtol=1e-5, atol=1e-6, what="bank vs one rank over the concatenated batch")
        if world == 1:   # a one-rank exchange reproduces the single-GPU fold bit for bit
            assert torch.equal(sums0, s1)


def test_peer_exchange_reports_a_missing_send(dev):
    """A consumer whose vectors never arrive must give up after its bounded poll (2 s) and flag status bit 8 -- an error
    code, not a hung GPU."""
    from uemda_b200.exchange import PeerExchange
    xs = PeerExchange.local_only(2, 3, 64, depth=2, device=dev)
    bank = torch.zeros(3, 64, device=dev)
    xs[0].fold_finalize(0, bank, decay=0.9)
    assert xs[0].status() & 8


def test_l2_hint_options_do_not_change_results(dev):
    """The L2 eviction-priority hints (uem_set_option l2_*) only steer cache replacement: every output of the fused chain
    and of the source-side prototype statistics is bit-identical with every combination of them."""
    from uemda_b200 import _lib, mining, ops
    from uemda_b200.gast.alignment import DownscaleLabel
    b, c, H, W, h, w, k = 2, 6, 128, 256, 8, 16, 64
    g = torch.Generator().manual_seed(77)
    soft = torch.softmax(torch.randn(b, c, H, W, generator=g) * 3, dim=1).to(dev)
    sup = torch.randint(0, 53, (b, 1, H, W), generator=g).to(dev)
    feat = torch.randn(b, k, h, w, generator=g).to(dev)
    protos = torch.randn(c, k, generator=g).to(dev)
    p1 = (torch.randn(b, c, h, w, generator=g) * 4).to(dev)
    p2 = (torch.randn(b, c, h, w, generator=g) * 4).to(dev)
    label_s = torch.randint(-1, c, (b, H, W), generator=g).to(dev)
    down = DownscaleLabel(16, c, -1, 0.75)
    lib = _lib.load()
    defaults = {"l2_stream": 1, "l2_last_use": 1, "l2_region": 1, "l2_keep": 0}
    combos = [dict(defaults), {"l2_stream": 0, "l2_last_use": 0, "l2_region": 0, "l2_keep": 0},
              {"l2_stream": 1, "l2_last_use": 0, "l2_region": 2, "l2_keep": 2}]
    outs = []
    try:
        for combo in combos:
            for name, v in combo.items():
                _lib.check(lib.uem_set_option(name.encode(), v))
            res = mining.refine_select(7, soft, 2.0, feat=feat, prototypes=protos, pred1=p1, pred2=p2, sup=sup,
                                       select=(0.8, 0.6, -1), uvem=(0.2, 0.7, 4.0))
            sums, counts = ops.proto_accumulate(feat, down(label_s), c)
            outs.append([t.clone() for t in res if t is not None] + [sums.clone(), counts.clone()])
    finally:
        for name, v in defaults.items():
            lib.uem_set_option(name.encode(), v)
    for other in outs[1:]:
        assert len(other) == len(outs[0])
        for a, b2 in zip(outs[0], other):
            bits = torch.int32 if a.dtype == torch.float32 else a.dtype   # bit patterns: NaN-safe
            assert torch.equal(a.view(bits), b2.view(bits))


# ------------------------------------------------------------------------------------ f4: IAST thresholds, sliding windows
def test_iast_golden_thresholds_and_labels(dev):
    """IAST class-wise percentile thresholds + thresholded labels against the reference's own ias_thresh driven through the
    per-batch body of generate_pseudo (tests/golden/iast_small.npz): thresholds (float64 state and the float32 percentile)
    and uint8 label maps bit for bit over three chained batches, one of them with a class that (almost) never wins."""
    import os
    from uemda_b200.utils.tools import IASTSelector
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "iast_small.npz"))
    alpha, beta, gamma = [float(v) for v in z["iast_params"]]
    sel = IASTSelector(n_class=z["in_probs_0"].shape[1], pl_alpha=alpha, pl_beta=beta, pl_gamma=gamma, device=dev)
    for step in range(3):
        assert np.array_equal(sel.cls_thresh.cpu().numpy(), z["in_thresh_%d" % step]), "threshold state entering batch %d" % step
        labels = sel.step(torch.from_numpy(z["in_probs_%d" % step]).to(dev))
        assert np.array_equal(sel.tmp_thresh.cpu().numpy(), z["out_tmp_thresh_%d" % step]), "percentiles of batch %d" % step
        assert np.array_equal(sel.cls_thresh.cpu().numpy(), z["out_thresh_%d" % step]), "thresholds after batch %d" % step
        assert np.array_equal(labels.cpu().numpy(), z["out_labels_%d" % step]), "labels of batch %d" % step


@pytest.mark.parametrize("shape,scale", [((2, 7, 96, 128), 3.0), ((1, 6, 33, 47), 1.0), ((4, 3, 64, 64), 8.0), ((8, 6, 512, 512), 2.0)])
def test_iast_vs_oracle_shapes(dev, shape, scale):
    """The same against the oracle restatement (np.percentile over float16 lists) at ragged and full config-2 shapes, two
    chained batches; per-class sample counts equal the argmax histogram."""
    from oracle import uem_oracle as O
    from uemda_b200.utils.tools import IASTSelector
    b, c, H, W = shape
    g = torch.Generator().manual_seed(b * 100 + W)
    sel = IASTSelector(n_class=c, pl_alpha=0.2, pl_beta=0.9, pl_gamma=8.0, device=dev)
    thr = np.ones(c) * 0.9
    for step in range(2):
        probs = torch.softmax(torch.randn(b, c, H, W, generator=g) * scale, dim=1)
        thr, want = O.iast_batch_step(probs, thr, 0.2, 0.9, 8.0)
        got = sel.step(probs.to(dev))
        assert np.array_equal(sel.cls_thresh.cpu().numpy(), thr), "thresholds, batch %d: %s vs %s" % (step, sel.cls_thresh.cpu().numpy(), thr)
        assert np.array_equal(got.cpu().numpy(), want), "labels, batch %d" % step
        assert np.array_equal(sel.counts.cpu().numpy(), np.bincount(probs.argmax(dim=1).reshape(-1).numpy(), minlength=c))


def test_sliding_window_golden(dev):
    """pre_slide (tools.py:61-97) against the reference's own run with a stand-in model that replays the golden tiles."""
    import os
    from uemda_b200.utils import tools as T
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "iast_small.npz"))
    H, W, th, tw = [int(v) for v in z["slide_meta"]]
    tiles = [torch.from_numpy(t).to(dev) for t in z["slide_tiles"]]
    it = iter(tiles)
    image = torch.zeros(tiles[0].shape[0], 3, H, W, device=dev)
    full = T.pre_slide(lambda x: next(it), image, num_classes=tiles[0].shape[1], tile_size=(th, tw), tta=False)
    _eq(full, torch.from_numpy(z["slide_out"]), "pre_slide")
    # TTA mean: 8 views of a model that is equivariant (identity) average back to the input
    x = torch.rand(1, 4, 32, 32, device=dev)
    assert_close(T.tta_predict(lambda a: a, x), x, rtol=1e-6, atol=1e-7, what="tta of the identity")
    from oracle import uem_oracle as O
    views = [torch.rand(1, 4, 16, 16) for _ in range(8)]
    assert_close(T.views_mean([v.to(dev) for v in views]), O.tta_mean(views), rtol=1e-6, atol=1e-7, what="views mean")


def test_regeneration_label_histogram(dev):
    """run_sharded on one rank: the label histogram it returns counts every produced uint8 value exactly once."""
    from uemda_b200.gast.alignment import Aligner
    from uemda_b200.regen import PseudoLabelRegenerator
    from uemda_b200.synth import Workload, make_inputs
    wl = Workload("regen3", 2, 6, 64, 64, 32, 16, 16)
    batches, outs = [], []
    for i in range(3):
        inp = make_inputs(wl, seed=200 + i, with_source=False)
        batches.append({"soft": inp["soft"].pin_memory(), "sup": inp["sup"].pin_memory(), "feat": inp["feat"].pin_memory(),
                        "preds": [inp["pred1"].pin_memory(), inp["pred2"].pin_memory()], "names": None})
    al = Aligner(_Log(), feat_channels=wl.k, class_num=wl.c, decay=0.996)
    al.prototypes = inp["prototypes"].to(dev)
    regen = PseudoLabelRegenerator(al, 0.8, 0.6, mode="all", temp=2.0, num_regions=int(inp["ignore_id"]) + 1)
    n, hist = regen.run_sharded(batches, lambda names, arr: outs.append(arr.copy()), device=dev)
    assert n == 6
    want = np.bincount(np.concatenate([o.reshape(-1) for o in outs]), minlength=wl.c + 1)
    assert np.array_equal(hist.cpu().numpy(), want)


@pytest.mark.parametrize("shape", [(2, 6, 8, 8, 128, 128), (1, 7, 5, 9, 37, 50), (2, 3, 4, 4, 4, 4), (1, 8, 3, 5, 48, 80), (8, 6, 32, 32, 512, 512)])
@pytest.mark.parametrize("heads", [1, 2])
def test_uvem_loss_backward_matches_autograd(dev, shape, heads):
    """The fused UVEM-loss backward (per-block partials + fixed-order gather) against CPU autograd in float64 of
    scale * sum_px coef * CE(upsample(x_m))[target], up-sampled as the reference does (bilinear, align_corners), up to
    fp32 summation order; and bit-reproducible run to run."""
    import torch.nn.functional as F
    from oracle import uem_oracle as O
    from uemda_b200 import ops
    b, c, h, w, H, W = shape
    g = torch.Generator().manual_seed(H * 7 + W)
    x1 = (torch.randn(b, c, h, w, generator=g) * 3).to(dev)
    x2 = (torch.randn(b, c, h, w, generator=g) * 3).to(dev) if heads == 2 else None
    target = torch.randint(-1, c, (b, H, W), generator=g).to(dev)
    coef = torch.rand(b * H * W, generator=g).to(dev)
    coef[target.reshape(-1) < 0] = 0.0
    coef[torch.rand(b * H * W, generator=g).to(dev) < 0.3] = 0.0
    scale = torch.tensor([0.37], device=dev)
    a = ops.uvem_loss_backward(x1, x2, target, coef, scale)
    a2 = ops.uvem_loss_backward(x1, x2, target, coef, scale)
    cf = coef.cpu().double().reshape(b, H, W)
    for m, x in enumerate((x1, x2)[:heads]):
        assert torch.equal(a[m], a2[m]), "backward is not bit-reproducible"
        xd = x.cpu().double().requires_grad_(True)
        ce = F.cross_entropy(O.upsample_bilinear(xd, (H, W)), target.cpu(), reduction="none", ignore_index=-1)
        (ce * cf).sum().backward()
        r = xd.grad * float(scale)
        tol = 1e-5 * float(r.abs().max())
        assert_close(a[m], r, rtol=1e-4, atol=tol, what="backward vs autograd, head %d" % m)


def test_bucketize_matches_torch(dev):
    """a15 companion: torch.bucketize over the 31 edges of the GHM / GDP gradient-norm bins (balance.py:194,263),
    including values on the edges, outside [0, 1], the -1 marker of ignored pixels, NaN and infinities."""
    from uemda_b200 import ops
    g = torch.Generator().manual_seed(9)
    edges = torch.arange(31).float() / 30
    x = torch.cat([torch.rand(100000, generator=g) * 1.4 - 0.2, edges, torch.tensor([-1.0, float("nan"), float("inf"), -float("inf")])])
    _eq(ops.bucketize(x.to(dev), edges.to(dev)), torch.bucketize(x, edges), "bucketize")
    _eq(ops.bucketize(x.reshape(-1, 5)[:100].to(dev), edges.to(dev)), torch.bucketize(x.reshape(-1, 5)[:100], edges), "bucketize 2-d")


def test_peer_exchange_merged_launch_world_of_one(dev):
    """The merged send + poll + fold + EMA launch (uem_xchg_exchange_fold_ema_f32) in a world of one rank (on real ranks
    every launch must run while the others run, so more ranks cannot be emulated in sequence on one device; bench.py
    --gpus N checks them against a one-GPU run): bit-equal to the plain image-order fold + EMA, over slot reuse."""
    from uemda_b200 import ops
    from uemda_b200.exchange import PeerExchange
    c, k, h, w, b = 6, 256, 8, 8, 3
    g = torch.Generator().manual_seed(4)
    x = PeerExchange.local_only(1, c, k, depth=3, device=dev)[0]
    bank = torch.randn(c, k, generator=g).to(dev)
    ref = bank.clone()
    gid = torch.zeros(1, dtype=torch.int64, device=dev)
    for step in range(7):
        slot = step % 3
        feat = torch.randn(b, k, h, w, generator=g).to(dev)
        lab = torch.randint(-1, c if step != 2 else 3, (b, 1, h, w), generator=g).to(dev)
        mid = torch.randint(0, 1 << 33, (1,), generator=g).to(dev)
        hist = ops.class_hist(lab, c)
        part = ops.proto_accumulate(feat, lab, c, -1, fold=False)
        x.send(None, mid, slot, global_id_out=gid, part="id")
        _, sums, counts, hout = x.exchange_fold(part, slot, bank, decay=0.9, out=bank, hist=hist, want_sums=True, want_hist=True)
        assert x.status() == 0 and int(gid) == int(mid)
        s1, n1 = ops.proto_accumulate(feat, lab, c, -1)
        assert torch.equal(sums, s1)
        _eq(counts, n1, "counts")
        _eq(hout, hist, "histogram")
        _, ref = ops.proto_finalize(s1, n1, ref, decay=0.9, want_local=False)
        assert torch.equal(bank, ref), "merged exchange launch differs from fold + EMA at step %d" % step
