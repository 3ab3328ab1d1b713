#!/usr/bin/env python
"""Development aid: per-CTA timeline of the fused refine kernel (library built with -DUEM_REFINE_TIMING, --tag=t).
Stamps (%globaltimer, ns) per CTA: 0 entry, 1 dependency wait + ignored id, 2 first setup done, 3 first row landed,
4 first row done, 5 last row done, 6 statistics flushed."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("UEM_B200_LIB", os.path.join(ROOT, "uemda_b200", "libuem_b200_t.so"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from uemda_b200 import _lib, config, ops  # noqa: E402
from uemda_b200.synth import WORKLOADS, make_inputs  # noqa: E402


def main():
    wl = WORKLOADS[sys.argv[1] if len(sys.argv) > 1 else "cfg2_isprs_8x6x512"]
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    config.strict_asserts = False
    inp = make_inputs(wl, seed=2333)
    sets = [{k: torch.roll(inp[k], i, 0).to(dev) for k in ("soft", "sup", "feat", "pred1", "pred2")} for i in range(3)]
    protos = inp["prototypes"].to(dev)
    R = int(inp["ignore_id"]) + 1
    for s in sets:
        s["simi"] = ops.pearson_dist_nchw(s["feat"], protos, reciprocal=True)
        s["rmax"] = ops.region_reduce(s["soft"], s["sup"], "max", dim_size=R, planar=True)
        s["ign"] = ops.i64_minmax(s["sup"])[1:].clone()
    fn = lambda s: ops.label_refine(7, s["soft"], 2.0, simi=s["simi"], pred1=s["pred1"], pred2=s["pred2"], sup=s["sup"],  # noqa: E731
                                    region_max=s["rmax"], ignored_id=s["ign"])
    for i in range(6):
        fn(sets[i % 3])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn(sets[0])
    e1.record()
    torch.cuda.synchronize()
    buf = (ctypes.c_ulonglong * (1024 * 8))()
    dbg = lib.__getattr__("uem_debug_refine_timing")
    dbg.restype = ctypes.c_int
    dbg(buf)
    t = np.frombuffer(buf, dtype=np.uint64).reshape(1024, 8).astype(np.int64)
    t = t[t[:, 0] > 0]
    t0 = t[:, 0].min()
    rel = (t - t0) / 1e3
    print("CTAs %d; event-timed launch (2 kernels: region weights + refine) %.1f us" % (len(t), e0.elapsed_time(e1) * 1e3))
    names = ["entry", "dep wait + ignored id", "first setup done", "first row landed", "first row done", "last row done", "stats flushed"]
    for i, nm in enumerate(names):
        c = rel[:, i]
        print("%-24s min %6.2f  median %6.2f  p95 %6.2f  max %6.2f us" % (nm, c.min(), np.median(c), np.percentile(c, 95), c.max()))
    life = rel[:, 6] - rel[:, 0]
    smid = t[:, 7]
    # where does the spread come from?  per-SM means (3 CTAs share an SM), per image, per strip
    by_sm = {}
    for sm, lf in zip(smid, life):
        by_sm.setdefault(int(sm), []).append(lf)
    sm_mean = np.array([np.mean(v) for v in by_sm.values()])
    within = np.mean([np.max(v) - np.min(v) for v in by_sm.values() if len(v) > 1])
    print("per-SM mean lifetime: min %.2f max %.2f std %.2f us; mean spread WITHIN an SM %.2f us; SMs used %d" % (
        sm_mean.min(), sm_mean.max(), sm_mean.std(), within, len(by_sm)))
    n = len(life)
    img = (np.arange(n) * wl.b // n)
    print("per-image mean lifetime:", " ".join("%.1f" % life[img == i].mean() for i in range(wl.b)))
    order = np.argsort(life)
    print("slowest 12 CTAs (blockIdx, smid, us):", [(int(i), int(smid[i]), round(float(life[i]), 1)) for i in order[-12:]])
    print("fastest 12 CTAs (blockIdx, smid, us):", [(int(i), int(smid[i]), round(float(life[i]), 1)) for i in order[:12]])
    rows = rel[:, 5] - rel[:, 4]
    print("corr(lifetime, blockIdx) %.2f; corr(lifetime, smid) %.2f" % (np.corrcoef(life, np.arange(n))[0, 1], np.corrcoef(life, smid)[0, 1]))
    print("CTA lifetime: min %.2f median %.2f max %.2f us; rows phase (first row done -> last row done) median %.2f us" % (
        life.min(), np.median(life), life.max(), np.median(rel[:, 5] - rel[:, 4])))


if __name__ == "__main__":
    main()
