"""Functional wrappers: torch CUDA tensors in, torch CUDA tensors out, one C-ABI call each.

All arithmetic happens in libuem_b200.so (hand-written sm_100a kernels); torch is used only to
allocate outputs/workspaces and to hand over raw pointers and the current stream.  Inputs are never
mutated; outputs are fresh tensors on the input's device, detached from autograd.
"""
import math
import struct

import torch

from . import _lib as L
from . import config

VIEW_PROTO, VIEW_PRED, VIEW_SUP = 1, 2, 4
VIEW_REGIONS_READY = 8  # uem_mine_refine_select_f32 only: mining.region_phase already ran on the workspace
VIEW_SIMI_READY = 16    # uem_mine_refine_select_f32 only: mining.proto_phase already ran on the workspace
REDUCE = {"sum": 0, "add": 0, "max": 1, "mean": 2}
MODE_VIEWS = {"all": VIEW_PROTO | VIEW_PRED | VIEW_SUP, "p": VIEW_PROTO, "l": VIEW_PRED, "s": VIEW_SUP}


def f32(x):
    """Python double -> nearest fp32 (what torch does to a Python scalar operand of an fp32 tensor)."""
    return struct.unpack("f", struct.pack("f", float(x)))[0]


# --------------------------------------------------------------------------------------------- a1-a4
def softmax_conf_entropy_argmax(x1, x2=None, size=None, temp=1.0, want=("soft", "conf", "entropy", "argmax")):
    """tools/train_align_uem.py:158-160 fused with max/argmax/entropy.  x1,x2 (b,c,h,w) logits."""
    L.require_cuda(x1, x2)
    x1 = L.f32c(x1.detach())
    x2 = None if x2 is None else L.f32c(x2.detach())
    b, c, h, w = x1.shape
    H, W = (h, w) if size is None else (int(size[0]), int(size[1]))
    lib = L.bind(x1)
    out = {}
    out["soft"] = torch.empty((b, c, H, W), dtype=torch.float32, device=x1.device) if "soft" in want else None
    out["conf"] = torch.empty((b, H, W), dtype=torch.float32, device=x1.device) if "conf" in want else None
    out["entropy"] = torch.empty((b, H, W), dtype=torch.float32, device=x1.device) if "entropy" in want else None
    out["argmax"] = torch.empty((b, H, W), dtype=torch.int64, device=x1.device) if "argmax" in want else None
    L.check(lib.uem_softmax_conf_entropy_argmax_f32(L.ptr(x1), L.ptr(x2), b, c, h, w, H, W, f32(temp), L.ptr(out["soft"]),
                                                    L.ptr(out["conf"]), L.ptr(out["entropy"]), L.ptr(out["argmax"]),
                                                    L.stream_of(x1)))
    return out


def _uvem_coefs(m, t, gamma):
    # balance.py:402-416: coefficients are Python doubles, rounded to fp32 when applied to fp32 tensors
    cl = f32(-1 / (m ** 2)) if m > 0 else 0.0
    cr = f32(-1 / ((t - m) ** 2)) if m < t else 0.0
    return f32(m), f32(t), f32(1.0 / gamma), cl, cr


def entropy_uvem_weight(soft, m=None, t=None, gamma=None, want_entropy=True):
    """balance.py:368-372 entropy of (b,c,H,W) probabilities (-> (b*H*W,)), optionally with get_weight."""
    L.require_cuda(soft)
    soft = L.f32c(soft.detach())
    b, c = soft.shape[:2]
    hw = soft[0, 0].numel()
    lib = L.bind(soft)
    ent = torch.empty(b * hw, dtype=torch.float32, device=soft.device) if want_entropy else None
    wgt = None
    if m is not None:
        wgt = torch.empty(b * hw, dtype=torch.float32, device=soft.device)
        mf, tf, ig, cl, cr = _uvem_coefs(m, t, gamma)
    else:
        mf, tf, ig, cl, cr = 0.0, 1.0, 1.0, 0.0, 0.0
    L.check(lib.uem_entropy_uvem_weight_f32(L.ptr(soft), b, c, hw, mf, tf, ig, cl, cr, L.ptr(ent), L.ptr(wgt), L.stream_of(soft)))
    return ent, wgt


def uvem_weight(u, m, t, gamma):
    """UVEMLoss.get_weight, balance.py:396-423."""
    L.require_cuda(u)
    uc = L.f32c(u.detach())
    lib = L.bind(uc)
    out = torch.empty_like(uc)
    mf, tf, ig, cl, cr = _uvem_coefs(m, t, gamma)
    L.check(lib.uem_uvem_weight_f32(L.ptr(uc), uc.numel(), mf, tf, ig, cl, cr, L.ptr(out), L.stream_of(uc)))
    return out


def uvem_terms(soft, target, m, t, gamma, use_weight=True, ignore_label=-1):
    """Detached factors of UVEMLoss/UPSLoss.forward (balance.py:372-382): weight (n,), gate (n,) bool, valid count."""
    L.require_cuda(soft, target)
    soft = L.f32c(soft.detach())
    target = L.i64c(target.detach()).reshape(-1)
    b, c = soft.shape[:2]
    hw = soft[0, 0].numel()
    assert target.numel() == b * hw
    lib = L.bind(soft)
    wgt = torch.empty(b * hw, dtype=torch.float32, device=soft.device)
    gate = torch.empty(b * hw, dtype=torch.uint8, device=soft.device)
    valid = torch.zeros(1, dtype=torch.int64, device=soft.device)
    if use_weight:
        mf, tf, ig, cl, cr = _uvem_coefs(m, t, gamma)
    else:
        mf, tf, ig, cl, cr = 0.0, f32(t), 1.0, 0.0, 0.0
    L.check(lib.uem_uvem_terms_f32(L.ptr(soft), L.ptr(target), b, c, hw, mf, tf, ig, cl, cr, int(bool(use_weight)),
                                   int(ignore_label), L.ptr(wgt), L.ptr(gate), L.ptr(valid), L.stream_of(soft)))
    return wgt, gate.bool(), valid


# --------------------------------------------------------------------------------------------- a5
def class_max(mask):
    """per-(b,c) max and min over pixels; (b,c,H,W) -> (b,c), (b,c), has_nan (1,) int32."""
    L.require_cuda(mask)
    mask = L.f32c(mask.detach())
    b, c = mask.shape[:2]
    hw = mask[0, 0].numel()
    lib = L.bind(mask)
    cmax = torch.empty((b, c), dtype=torch.float32, device=mask.device)
    cmin = torch.empty((b, c), dtype=torch.float32, device=mask.device)
    nan = torch.zeros(1, dtype=torch.int32, device=mask.device)
    ws = L.workspace(lib.uem_class_max_ws_bytes(b, c, hw), mask)
    L.check(lib.uem_class_max_f32(L.ptr(mask), b, c, hw, L.ptr(cmax), L.ptr(cmin), L.ptr(nan), L.ptr(ws), L.stream_of(mask)))
    return cmax, cmin, nan


def pseudo_select(mask, cmax, cutoff_top, cutoff_low, ignore_label=-1, variant=0):
    L.require_cuda(mask, cmax)
    mask = L.f32c(mask.detach())
    b, c, h, w = mask.shape
    lib = L.bind(mask)
    out = torch.empty((b, h, w), dtype=torch.int64, device=mask.device)
    L.check(lib.uem_pseudo_select_f32(L.ptr(mask), L.ptr(cmax), b, c, h * w, f32(cutoff_top), f32(cutoff_low),
                                      int(ignore_label), int(variant), L.ptr(out), L.stream_of(mask)))
    return out


def pseudo_select_stats(mask, stats, cutoff_top, cutoff_low, ignore_label=-1, uvem=None, want_entropy=False):
    """pseudo_selection fed by the (b, c+2) uint32 class-statistics table the refine kernel raised; with
    ``uvem=(m, t, gamma)`` / ``want_entropy`` also the entropy and UVEM weight of the same pass.
    Returns hard, or (hard, entropy|None, weight|None)."""
    import ctypes
    L.require_cuda(mask, stats)
    mask = L.f32c(mask.detach())
    b, c, h, w = mask.shape
    lib = L.bind(mask)
    out = torch.empty((b, h, w), dtype=torch.int64, device=mask.device)
    extra = want_entropy or uvem is not None
    ent = torch.empty(b * h * w, dtype=torch.float32, device=mask.device) if extra else None
    wgt = torch.empty(b * h * w, dtype=torch.float32, device=mask.device) if uvem is not None else None
    uv = (ctypes.c_float * 5)(*_uvem_coefs(*uvem)) if uvem is not None else None
    L.check(lib.uem_select_entropy_stats_f32(L.ptr(mask), L.ptr(stats), b, c, h * w, f32(cutoff_top), f32(cutoff_low),
                                             int(ignore_label), L.ptr(out), uv, L.ptr(ent), L.ptr(wgt), L.stream_of(mask)))
    return (out, ent, wgt) if extra else out


def class_stats_decode(stats, c):
    """(b, c+2) uint32 statistics table -> cmax (b,c) fp32, image_min (b,) fp32 (NaN where the bad flag is set)."""
    L.require_cuda(stats)
    b = stats.shape[0]
    lib = L.bind(stats)
    cmax = torch.empty((b, c), dtype=torch.float32, device=stats.device)
    imin = torch.empty((b,), dtype=torch.float32, device=stats.device)
    L.check(lib.uem_class_stats_decode_f32(L.ptr(stats), b, c, L.ptr(cmax), L.ptr(imin), L.stream_of(stats)))
    return cmax, imin


# --------------------------------------------------------------------------------------------- seam
def i64_minmax(x):
    """(2,) int64 device tensor [min, max] -- no host sync."""
    L.require_cuda(x)
    x = L.i64c(x.detach())
    lib = L.bind(x)
    out = torch.empty(2, dtype=torch.int64, device=x.device)
    L.check(lib.uem_i64_minmax(L.ptr(x), x.numel(), L.ptr(out), L.stream_of(x)))
    return out


def region_reduce(src, index, reduce="sum", dim_size=None, planar=False):
    """Segmented reduction over region ids (the torch_scatter.scatter seam, dim=1).

    src: (b,N,c) [planar=False] or an NCHW map (b,c,*spatial) [planar=True, read in place];
    index: (b,N) / (b,N,1) / (b,1,H,W) int64.  Returns (b,R,c) with R = index.max()+1 (one host sync,
    exactly like torch_scatter) unless dim_size is given."""
    L.require_cuda(src, index)
    index = L.i64c(index.detach())
    b = index.shape[0]
    idx = index.reshape(b, -1)
    N = idx.shape[1]
    is_float = src.is_floating_point()
    src = L.f32c(src.detach()) if is_float else L.i64c(src.detach())
    if planar:
        c = src.shape[1]
        assert src[0, 0].numel() == N
        strides = (c * N, 1, N)
    else:
        assert src.dim() == 3 and src.shape[1] == N
        c = src.shape[2]
        strides = (N * c, c, 1)
    lib = L.bind(src)
    if dim_size is None:
        dim_size = int(i64_minmax(idx)[1].item()) + 1
    R = int(dim_size)
    op = REDUCE[reduce]
    if is_float:
        out = torch.empty((b, R, c), dtype=torch.float32, device=src.device)
        ws = L.workspace(lib.uem_region_reduce_ws_bytes(b, R, c), src)
        L.check(lib.uem_region_reduce_f32(L.ptr(src), strides[0], strides[1], strides[2], L.ptr(idx), b, N, c, R, op,
                                          L.ptr(out), L.ptr(ws), L.stream_of(src)))
    else:
        if reduce == "mean":
            raise NotImplementedError("integer mean is not used by the reference (alignment.py:187 is 'sum')")
        out = torch.empty((b, R, c), dtype=torch.int64, device=src.device)
        L.check(lib.uem_region_reduce_i64(L.ptr(src), strides[0], strides[1], strides[2], L.ptr(idx), b, N, c, R, op,
                                          L.ptr(out), None, L.stream_of(src)))
    return out


def superpixel_expand(hard, sup, class_num, ignore_label=-1, num_regions=None):
    """alignment.py:175-192.  hard (b,H,W), sup (b,1,H,W) -> (b,H,W) int64."""
    L.require_cuda(hard, sup)
    hard = L.i64c(hard.detach())
    sup = L.i64c(sup.detach())
    b = hard.shape[0]
    N = hard[0].numel()
    assert sup.numel() == b * N
    lib = L.bind(hard)
    R = int(i64_minmax(sup)[1].item()) + 1 if num_regions is None else int(num_regions)
    out = torch.empty_like(hard)
    ws = L.workspace(lib.uem_superpixel_expand_ws_bytes(b, R, class_num), hard)
    L.check(lib.uem_superpixel_expand_i64(L.ptr(hard), L.ptr(sup), b, N, class_num, R, int(ignore_label), L.ptr(out),
                                          L.ptr(ws), L.stream_of(hard)))
    if config.strict_asserts:
        # status word behind [counts | winner] (uem_region.cu): pixels with an id outside [0,R) or a label outside
        # {ignore} U [0,c) were skipped; the reference's one_hot / scatter / gather raise on them (alignment.py:184-190)
        off = (b * R * class_num + b * R) * 4
        bits = int(ws[off:off + 4].view(torch.int32).item())
        if bits & 1:
            raise RuntimeError("Class values must be non-negative and smaller than num_classes.")
        if bits & 2:
            raise RuntimeError("superpixel_expand: superpixel id outside [0, num_regions) (index out of bounds in the "
                               "reference's scatter/gather, alignment.py:187-190)")
    return out


# --------------------------------------------------------------------------------------------- a8
def downscale_label(label, scale_factor, n_classes, ignore_label=-1, min_ratio=0.75, status=None):
    """alignment.py:494-509.  (b,H,W)|(b,1,H,W) int64 -> (b,1,h,w) int64."""
    L.require_cuda(label)
    label = L.i64c(label.detach())
    if label.dim() == 4:
        label = label.squeeze(1)
    assert label.dim() == 3
    b, H, W = label.shape
    h, w = H // scale_factor, W // scale_factor
    lib = L.bind(label)
    out = torch.empty((b, 1, h, w), dtype=torch.int64, device=label.device)
    L.check(lib.uem_downscale_label_i64(L.ptr(label), b, H, W, int(scale_factor), int(n_classes), int(ignore_label),
                                        f32(min_ratio), L.ptr(out), L.ptr(status), L.stream_of(label)))
    return out


# --------------------------------------------------------------------------------------------- a9
def pearson_dist_nchw(feat, prototypes, eps=1e-7, reciprocal=False):
    """feat (b,k,h,w) read in place, prototypes (c,k) -> (b,c,h,w) distance (or 1/distance)."""
    L.require_cuda(feat, prototypes)
    feat = L.f32c(feat.detach())
    protos = L.f32c(prototypes.detach())
    b, k, h, w = feat.shape
    m = protos.shape[0]
    assert protos.shape[1] == k
    lib = L.bind(feat)
    out = torch.empty((b, m, h, w), dtype=torch.float32, device=feat.device)
    ws = L.workspace(lib.uem_pearson_nchw_ws_bytes(b, h * w, m, k), feat)
    L.check(lib.uem_pearson_dist_nchw_f32(L.ptr(feat), b, k, h * w, L.ptr(protos), m, f32(eps), int(reciprocal), L.ptr(out),
                                          L.ptr(ws), L.stream_of(feat)))
    return out


def pearson_dist_rows(feat1, feat2, eps=1e-7):
    """alignment.py:424-451.  (n,k),(m,k) -> (n,m)."""
    L.require_cuda(feat1, feat2)
    f1 = L.f32c(feat1.detach())
    f2 = L.f32c(feat2.detach())
    assert f1.shape[-1] == f2.shape[-1]
    n, k = f1.shape
    m = f2.shape[0]
    lib = L.bind(f1)
    out = torch.empty((n, m), dtype=torch.float32, device=f1.device)
    ws = L.workspace(lib.uem_pearson_ws_bytes(m, k), f1)
    L.check(lib.uem_pearson_dist_rows_f32(L.ptr(f1), n, k, L.ptr(f2), m, f32(eps), L.ptr(out), L.ptr(ws), L.stream_of(f1)))
    return out


# --------------------------------------------------------------------------------------------- a6
def label_refine(views, soft, temp, simi=None, pred1=None, pred2=None, sup=None, region_max=None, ignored_id=None,
                 want_stats=True):
    """One fused full-resolution kernel (alignment.py:215-292).  Returns (refined, class stats table|None)."""
    L.require_cuda(soft, simi, pred1, pred2, sup, region_max, ignored_id)
    soft = L.f32c(soft.detach())
    b, c, H, W = soft.shape
    lib = L.bind(soft)
    low = simi if simi is not None else pred1
    h, w = (low.shape[-2], low.shape[-1]) if low is not None else (0, 0)
    R = region_max.shape[1] if region_max is not None else 0
    out = torch.empty_like(soft)
    stats = torch.zeros((b, c + 2), dtype=torch.int32, device=soft.device) if want_stats else None
    ws = L.workspace(lib.uem_label_refine_ws_bytes(b, c, R, W), soft)
    L.check(lib.uem_label_refine_f32(int(views), L.ptr(simi), L.ptr(pred1), L.ptr(pred2), h, w, L.ptr(sup), L.ptr(region_max),
                                     R, L.ptr(ignored_id), L.ptr(soft), b, c, H, W, f32(temp), L.ptr(out), L.ptr(stats),
                                     L.ptr(ws), L.stream_of(soft)))
    return out, stats


def proto_weight_4pixel(simi, hard, ignore_label=-1, eps=1e-7):
    L.require_cuda(simi, hard)
    simi = L.f32c(simi)
    hard = L.i64c(hard.detach())
    b, c, h, w = simi.shape
    _, H, W = hard.shape
    lib = L.bind(simi)
    out = torch.empty(b * H * W, dtype=torch.float32, device=simi.device)
    L.check(lib.uem_proto_weight_4pixel_f32(L.ptr(simi), h, w, L.ptr(hard), b, c, H, W, int(ignore_label), f32(eps),
                                            L.ptr(out), L.stream_of(simi)))
    return out


# --------------------------------------------------------------------------------------------- a10-a12
def proto_accumulate(feat, label_down, class_num, ignore_label=-1, fold=True, ws=None):
    """Masked per-class feature sums (c,k) fp32 and counts (c,) int64 (alignment.py:341-348).
    fold=False: returns the opaque per-image partials (for proto_fold_finalize) instead.
    ws: optional preallocated scratch (``proto_accumulate_ws``): a static buffer when the partials cross CUDA graphs."""
    L.require_cuda(feat, label_down)
    feat = L.f32c(feat.detach())
    label = L.i64c(label_down.detach())
    b, k, h, w = feat.shape
    assert label.numel() == b * h * w, "label must be at feature resolution"
    lib = L.bind(feat)
    sums = torch.empty((class_num, k), dtype=torch.float32, device=feat.device) if fold else None
    counts = torch.empty((class_num,), dtype=torch.int64, device=feat.device) if fold else None
    need = lib.uem_proto_accum_ws_bytes(b, class_num, k)
    if ws is None:
        ws = L.workspace(need, feat)
    assert ws.numel() >= need and ws.device == feat.device
    L.check(lib.uem_proto_accum_nchw_f32(L.ptr(feat), b, k, h * w, L.ptr(label), class_num, int(ignore_label), L.ptr(sums),
                                         L.ptr(counts), L.ptr(ws), L.stream_of(feat)))
    if not fold:
        return ws, (b, class_num, k)
    return sums, counts


def proto_accumulate_ws(b, class_num, k, device):
    """Scratch of proto_accumulate for a (b, k, h, w) feature map (holds the per-image partial sums and counts)."""
    return torch.empty(max(int(L.load().uem_proto_accum_ws_bytes(b, class_num, k)), 16), dtype=torch.uint8, device=device)


def proto_fold_finalize(partials, proto_old, eps=1e-7, decay=0.999, out=None):
    """partials from proto_accumulate(fold=False) -> EMA-updated prototypes in one launch (alignment.py:347-353,463-466).
    out may be ``proto_old`` itself."""
    ws, (b, c, k) = partials
    L.require_cuda(ws, proto_old)
    lib = L.bind(ws)
    proto_old = L.f32c(proto_old.detach())
    new = out if out is not None else torch.empty_like(proto_old)
    L.check(lib.uem_proto_fold_finalize_ema_f32(L.ptr(ws), b, c, k, L.ptr(proto_old), f32(eps), f32(1.0 - decay), f32(decay),
                                                L.ptr(new), L.stream_of(ws)))
    return new


def proto_accumulate_soft(feat, soft):
    """sum over pixels of feat * bilinear_down(soft) -> (c,k) (alignment.py:98-104 before the mean)."""
    L.require_cuda(feat, soft)
    feat = L.f32c(feat.detach())
    soft = L.f32c(soft.detach())
    b, k, h, w = feat.shape
    _, c, H, W = soft.shape
    lib = L.bind(feat)
    sums = torch.empty((c, k), dtype=torch.float32, device=feat.device)
    ws = L.workspace(lib.uem_proto_accum_soft_ws_bytes(b, c, k, h, w), feat)
    L.check(lib.uem_proto_accum_soft_f32(L.ptr(feat), b, k, h, w, L.ptr(soft), c, H, W, L.ptr(sums), L.ptr(ws), L.stream_of(feat)))
    return sums


def proto_finalize(sums, counts, proto_old, eps=1e-7, decay=None, mean_n=0, want_local=True, out=None):
    """local = sums/(cnt+eps) with the keep-old rule (or sums/mean_n), optional EMA. Returns (local, new).
    out: optional (c,k) fp32 tensor receiving the EMA result; may be ``proto_old`` itself (element-wise, in place)."""
    L.require_cuda(sums, counts, proto_old)
    c, k = sums.shape
    lib = L.bind(sums)
    proto_old = L.f32c(proto_old.detach())
    local = torch.empty_like(sums) if want_local else None
    new = (out if out is not None else torch.empty_like(sums)) if decay is not None else None
    omd, d = (f32(1.0 - decay), f32(decay)) if decay is not None else (0.0, 0.0)
    L.check(lib.uem_proto_finalize_ema_f32(L.ptr(sums), L.ptr(counts), int(mean_n), L.ptr(proto_old), c, k, f32(eps), omd, d,
                                           L.ptr(local), L.ptr(new), L.stream_of(sums)))
    return local, new


# --------------------------------------------------------------------------------------------- a14/a15
def class_hist(label, class_num, ignore_label=-1):
    """(c+1,) int64: per-class counts and, last, the number of non-ignored labels (balance.py:45-52)."""
    L.require_cuda(label)
    label = L.i64c(label.detach()).reshape(-1)
    lib = L.bind(label)
    hist = torch.zeros(class_num + 1, dtype=torch.int64, device=label.device)
    L.check(lib.uem_class_hist_i64(L.ptr(label), label.numel(), class_num, int(ignore_label), L.ptr(hist), L.stream_of(label)))
    return hist


def class_weight_lookup(label, table, ignore_label=-1):
    L.require_cuda(label, table)
    label = L.i64c(label.detach()).reshape(-1)
    table = L.f32c(table.detach())
    lib = L.bind(label)
    out = torch.empty(label.numel(), dtype=torch.float32, device=label.device)
    L.check(lib.uem_class_weight_lookup_f32(L.ptr(label), label.numel(), table.numel(), int(ignore_label), L.ptr(table),
                                            L.ptr(out), L.stream_of(label)))
    return out


def hist_f32(x, bins, lo, hi):
    """torch.histc(x, bins, lo, hi) as int64 counts (balance.py:193)."""
    L.require_cuda(x)
    x = L.f32c(x.detach()).reshape(-1)
    lib = L.bind(x)
    hist = torch.zeros(bins, dtype=torch.int64, device=x.device)
    L.check(lib.uem_hist_f32(L.ptr(x), x.numel(), int(bins), f32(lo), f32(hi), L.ptr(hist), L.stream_of(x)))
    return hist


def bucketize(x, boundaries):
    """torch.bucketize(x, boundaries) (right=False) as int64 (balance.py:194,263: gradient-norm bins of GHM / GDP)."""
    L.require_cuda(x, boundaries)
    shape = x.shape
    x = L.f32c(x.detach()).reshape(-1)
    boundaries = L.f32c(boundaries.detach()).reshape(-1)
    lib = L.bind(x)
    out = torch.empty(x.numel(), dtype=torch.int64, device=x.device)
    L.check(lib.uem_bucketize_f32(L.ptr(x), x.numel(), L.ptr(boundaries), boundaries.numel(), L.ptr(out), L.stream_of(x)))
    return out.reshape(shape)


# --------------------------------------------------------------------------------------------- regeneration
def label_plus1_u8(label):
    """uint8(label + 1): the on-disk form of a hard pseudo-label map (pseudo_generation.py:150-151)."""
    L.require_cuda(label)
    label = L.i64c(label.detach())
    lib = L.bind(label)
    out = torch.empty(label.shape, dtype=torch.uint8, device=label.device)
    L.check(lib.uem_label_plus1_u8_i64(L.ptr(label), label.numel(), L.ptr(out), L.stream_of(label)))
    return out


# --------------------------------------------------------------------------------------------- PCL loss (8f-2)
def pcl_forward(feat, prototypes, labels, temperature=8.0, ignore_label=-1):
    """uemda/loss.py:18-47 on an NCHW feature map read in place. Returns (loss (1,), coef (b,c+1,h*w), ws)."""
    L.require_cuda(feat, prototypes, labels)
    feat = L.f32c(feat.detach())
    protos = L.f32c(prototypes.detach())
    labels = L.i64c(labels.detach())
    b, k, h, w = feat.shape
    c = protos.shape[0]
    assert protos.shape[1] == k and labels.numel() == b * h * w
    lib = L.bind(feat)
    loss = torch.empty(1, dtype=torch.float32, device=feat.device)
    coef = torch.empty((b, c + 1, h * w), dtype=torch.float32, device=feat.device)
    ws = L.workspace(lib.uem_pcl_ws_bytes(b, k, h * w), feat)
    L.check(lib.uem_pcl_forward_f32(L.ptr(feat), b, k, h * w, L.ptr(protos), c, L.ptr(labels), int(ignore_label), f32(temperature),
                                    L.ptr(loss), L.ptr(coef), L.ptr(ws), L.stream_of(feat)))
    return loss, coef, ws


def pcl_backward(feat, coef, ws, grad_out=None):
    """d loss / d feat (b,k,h,w) from the coefficients of pcl_forward."""
    L.require_cuda(feat, coef, ws, grad_out)
    feat = L.f32c(feat.detach())
    b, k, h, w = feat.shape
    c = coef.shape[1] - 1
    lib = L.bind(feat)
    grad = torch.empty_like(feat)
    g = None if grad_out is None else L.f32c(grad_out.detach()).reshape(1)
    L.check(lib.uem_pcl_backward_f32(L.ptr(feat), b, k, h * w, c, L.ptr(coef), L.ptr(g), L.ptr(grad), L.ptr(ws), L.stream_of(feat)))
    return grad


# --------------------------------------------------------------------------------------------- f3
def uvem_loss_forward(x1, x2, target, coef):
    """sum_px coef * CE(upsample(x_m))[target] per head -> (heads,) float64 (balance.py:356-394, :437-457)."""
    L.require_cuda(x1, x2, target, coef)
    x1 = L.f32c(x1.detach())
    x2 = None if x2 is None else L.f32c(x2.detach())
    target = L.i64c(target.detach())
    coef = L.f32c(coef.detach()).reshape(-1)
    b, c, h, w = x1.shape
    H, W = target.shape[-2:]
    assert target.numel() == b * H * W and coef.numel() == b * H * W and (x2 is None or x2.shape == x1.shape)
    lib = L.bind(x1)
    sums = torch.zeros(2 if x2 is not None else 1, dtype=torch.float64, device=x1.device)
    L.check(lib.uem_uvem_loss_forward_f32(L.ptr(x1), L.ptr(x2), b, c, h, w, H, W, L.ptr(target), L.ptr(coef), L.ptr(sums),
                                          L.stream_of(x1)))
    return sums


def uvem_loss_backward(x1, x2, target, coef, scale):
    """scale * d/dx_m sum_px coef * CE(upsample(x_m))[target]; deterministic (no atomics)."""
    L.require_cuda(x1, x2, target, coef, scale)
    x1 = L.f32c(x1.detach())
    x2 = None if x2 is None else L.f32c(x2.detach())
    target = L.i64c(target.detach())
    coef = L.f32c(coef.detach()).reshape(-1)
    scale = L.f32c(scale.detach()).reshape(1)
    b, c, h, w = x1.shape
    H, W = target.shape[-2:]
    lib = L.bind(x1)
    g1 = torch.empty_like(x1)
    g2 = None if x2 is None else torch.empty_like(x2)
    ws = L.workspace(lib.uem_uvem_loss_backward_ws_bytes(b, c, h, w, 2 if x2 is not None else 1), x1)
    L.check(lib.uem_uvem_loss_backward_f32(L.ptr(x1), L.ptr(x2), b, c, h, w, H, W, L.ptr(target), L.ptr(coef), L.ptr(scale),
                                           L.ptr(g1), L.ptr(g2), L.ptr(ws), L.stream_of(x1)))
    return g1, g2


# --------------------------------------------------------------------------------------------- 8e
def pack_local(sums, counts, max_id, out=None):
    """[c*k sums | c counts | max id] -> (c*k+c+1,) float64 in one launch (the rank-local statistics of a step)."""
    L.require_cuda(sums, counts, max_id)
    sums = L.f32c(sums.detach())
    counts = L.i64c(counts.detach())
    max_id = L.i64c(max_id.detach()).reshape(-1)
    c, k = sums.shape
    lib = L.bind(sums)
    if out is None:
        out = torch.empty(c * k + c + 1, dtype=torch.float64, device=sums.device)
    assert out.dtype == torch.float64 and out.numel() == c * k + c + 1 and out.is_contiguous()
    L.check(lib.uem_pack_local_f64(L.ptr(sums), L.ptr(counts), L.ptr(max_id), c, k, L.ptr(out), L.stream_of(sums)))
    return out


def pack_local_partials(partials, max_id, out=None):
    """Per-image partials of proto_accumulate(fold=False) folded in image order and packed with the max id in one launch."""
    ws, (b, c, k) = partials
    L.require_cuda(ws, max_id)
    max_id = L.i64c(max_id.detach()).reshape(-1)
    lib = L.bind(ws)
    if out is None:
        out = torch.empty(c * k + c + 1, dtype=torch.float64, device=ws.device)
    assert out.dtype == torch.float64 and out.numel() == c * k + c + 1 and out.is_contiguous()
    L.check(lib.uem_pack_local_partials_f64(L.ptr(ws), b, c, k, L.ptr(max_id), L.ptr(out), L.stream_of(ws)))
    return out


def fold_gathered(gathered, c, k, out=None):
    """(world, c*k+c+1) float64 -> (sums (c,k) fp32, counts (c,) int64, max id (1,) int64), ranks folded in rank order.
    out: optional (sums, counts, max_id) tensors to write into (static buffers for CUDA-graph replay)."""
    L.require_cuda(gathered)
    assert gathered.dtype == torch.float64 and gathered.is_contiguous() and gathered.shape[1] == c * k + c + 1
    lib = L.bind(gathered)
    if out is not None:
        sums, counts, max_id = out
        assert sums.dtype == torch.float32 and sums.numel() == c * k and counts.dtype == torch.int64 and max_id.dtype == torch.int64
    else:
        sums = torch.empty((c, k), dtype=torch.float32, device=gathered.device)
        counts = torch.empty((c,), dtype=torch.int64, device=gathered.device)
        max_id = torch.empty((1,), dtype=torch.int64, device=gathered.device)
    L.check(lib.uem_fold_gathered_f64(L.ptr(gathered), gathered.shape[0], c, k, L.ptr(sums), L.ptr(counts), L.ptr(max_id),
                                      L.stream_of(gathered)))
    return sums, counts, max_id
