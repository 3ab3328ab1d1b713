#!/usr/bin/env python
"""Per-kernel device timing of the mining path at one workload (development aid, not the bench contract).

Every entry is captured into one CUDA graph per rotating input set (so Python launch overhead is out of the
picture), replayed back to back and timed with CUDA events; inputs rotate over --sets copies (cold L2 reads).
Prints us per call and algorithmic GB/s.
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from uemda_b200 import _lib, config, mining, ops  # noqa: E402
from uemda_b200.gast.alignment import DownscaleLabel  # noqa: E402
from uemda_b200.synth import WORKLOADS, make_inputs  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg2_isprs_8x6x512")
    ap.add_argument("--sets", type=int, default=3)
    ap.add_argument("--iters", type=int, default=60)
    ap.add_argument("--only", default="")
    ap.add_argument("--opt", action="append", default=[], help="name=value for uem_set_option (repeatable)")
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.load()
    for kv in args.opt:
        name, val = kv.split("=")
        _lib.check(_lib.load().uem_set_option(name.encode(), int(val)))
    config.strict_asserts = False
    inp = make_inputs(wl, seed=2333)
    keys = ("soft", "sup", "feat", "pred1", "pred2", "label_s", "feat_s")
    sets = [{k: torch.roll(inp[k], i, 0).to(dev) for k in keys} for i in range(args.sets)]
    protos = inp["prototypes"].to(dev)
    R = int(inp["ignore_id"]) + 1
    P = wl.pixels
    c = wl.c
    feat_bytes = wl.b * wl.k * wl.h * wl.w * 4
    down = DownscaleLabel(wl.scale, c, -1, 0.75)
    for s in sets:
        s["refined"], _ = mining.refine_select(7, s["soft"], 2.0, feat=s["feat"], prototypes=protos, pred1=s["pred1"],
                                               pred2=s["pred2"], sup=s["sup"], num_regions=R)
        s["stats"] = s["refined"]._uem_stats.stats
        s["hard"] = ops.pseudo_select_stats(s["refined"], s["stats"], 0.8, 0.6, -1)
        s["simi"] = ops.pearson_dist_nchw(s["feat"], protos, reciprocal=True)
        s["rmax"] = ops.region_reduce(s["soft"], s["sup"], "max", dim_size=R, planar=True)
        s["ign"] = ops.i64_minmax(s["sup"])[1:].clone()
        s["down"] = down(s["label_s"])
    ws = torch.zeros(_lib.load().uem_mine_ws_bytes(wl.b, c, wl.H, wl.W, wl.h, wl.w, wl.k, R), dtype=torch.uint8, device=dev)

    entries = {
        "pearson_nchw": (lambda s: ops.pearson_dist_nchw(s["feat"], protos, reciprocal=True), feat_bytes),
        "region_max": (lambda s: ops.region_reduce(s["soft"], s["sup"], "max", dim_size=R, planar=True), P * (4 * c + 8)),
        "i64_minmax": (lambda s: ops.i64_minmax(s["sup"]), P * 8),
        "label_refine": (lambda s: ops.label_refine(7, s["soft"], 2.0, simi=s["simi"], pred1=s["pred1"], pred2=s["pred2"],
                                                    sup=s["sup"], region_max=s["rmax"], ignored_id=s["ign"]), P * (8 * c + 8)),
        "select_stats": (lambda s: ops.pseudo_select_stats(s["refined"], s["stats"], 0.8, 0.6, -1, uvem=(0.2, 0.7, 4.0)),
                         P * (4 * c + 16)),
        "select_only": (lambda s: ops.pseudo_select_stats(s["refined"], s["stats"], 0.8, 0.6, -1), P * (4 * c + 8)),
        "class_max+select": (lambda s: ops.pseudo_select(s["refined"], ops.class_max(s["refined"])[0], 0.8, 0.6), P * (8 * c + 8)),
        "entropy_uvem": (lambda s: ops.entropy_uvem_weight(s["refined"], 0.2, 0.7, 4.0), P * (4 * c + 8)),
        "downscale": (lambda s: down(s["label_s"]), P * 8),
        "proto_accum": (lambda s: ops.proto_accumulate(s["feat_s"], s["down"], c), feat_bytes),
        "superpixel_expand": (lambda s: ops.superpixel_expand(s["hard"], s["sup"], c, num_regions=R), P * 24),
        "class_hist": (lambda s: ops.class_hist(s["hard"], c), P * 8),
        "logits_pass": (lambda s: ops.softmax_conf_entropy_argmax(s["pred1"], s["pred2"], size=(wl.H, wl.W)), P * (4 * c + 16)),
        "pcl_forward": (lambda s: ops.pcl_forward(s["feat_s"], protos, s["down"], 8.0), feat_bytes),
        "pcl_fwd+bwd": (lambda s: (lambda o: ops.pcl_backward(s["feat_s"], o[1], o[2]))(ops.pcl_forward(s["feat_s"], protos, s["down"], 8.0)),
                        3 * feat_bytes),
        "mine_chain": (lambda s: mining.refine_select(7, s["soft"], 2.0, feat=s["feat"], prototypes=protos, pred1=s["pred1"],
                                                      pred2=s["pred2"], sup=s["sup"], num_regions=R, select=(0.8, 0.6, -1),
                                                      ws=ws, uvem=(0.2, 0.7, 4.0)),
                       P * (8 * c + 8 + 8 + 4 * c + 8) + feat_bytes),
    }
    only = [x for x in args.only.split(",") if x]
    print("%-20s %10s %10s %8s" % ("entry", "us/call", "GB/s(alg)", "of 6537"))
    for name, (fn, nbytes) in entries.items():
        if only and name not in only:
            continue
        for s in sets:
            fn(s)
        torch.cuda.synchronize()
        # ONE graph holding `reps` back-to-back calls (rotating over the input sets): graph-launch latency on the host
        # (several us) would otherwise dominate the short kernels
        reps = 4 * len(sets)
        keep = []
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(reps):
                keep.append(fn(sets[i % len(sets)]))
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_rep = max(1, args.iters // reps)
        e0.record()
        for i in range(n_rep):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / (n_rep * reps)
        gbs = nbytes / us / 1e3
        print("%-20s %10.2f %10.1f %7.1f%%" % (name, us, gbs, 100 * gbs / 6536.7), flush=True)


if __name__ == "__main__":
    main()
