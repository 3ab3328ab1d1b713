#!/usr/bin/env python
"""Fused UVEM target loss (next row 8f-3) against the unfused drop-in path (PyTorch interpolate + cross_entropy + autograd)
at one workload: forward + backward, CUDA events, warm caches excluded by rotating over input sets."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn.functional as tnf  # noqa: E402

from uemda_b200 import _lib  # noqa: E402
from uemda_b200.gast.balance import UVEMLoss, loss_calc_uvem  # noqa: E402
from uemda_b200.synth import WORKLOADS, make_inputs  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg2_isprs_8x6x512")
    ap.add_argument("--iters", type=int, default=30)
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]
    dev = torch.device("cuda", 0)
    _lib.load()
    inp = make_inputs(wl, seed=2333)
    sets = []
    for i in range(3):
        soft = torch.roll(inp["soft"], i, 0).to(dev)
        sets.append({"soft": soft, "label": soft.argmax(1), "x1": torch.roll(inp["pred1"], i, 0).to(dev).requires_grad_(True),
                     "x2": torch.roll(inp["pred2"], i, 0).to(dev).requires_grad_(True)})
    fn = UVEMLoss(m=0.2, threshold=0.7, gamma=4.0, class_num=wl.c)

    def fused(s):
        loss = loss_calc_uvem([s["x1"], s["x2"]], s["label"], s["soft"], fn)
        loss.backward()
        return loss

    def unfused(s):
        up = [tnf.interpolate(x, size=s["label"].shape[-2:], mode="bilinear", align_corners=True) for x in (s["x1"], s["x2"])]
        loss = (fn(up[0], s["label"], s["soft"]) + fn(up[1], s["label"], s["soft"])) / 2
        loss.backward()
        return loss

    for name, f in (("fused fwd+bwd", fused), ("unfused fwd+bwd (PyTorch CE)", unfused)):
        for s in sets:
            f(s)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.iters):
            f(sets[i % 3])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.iters
        print("%-32s %8.3f ms/step  %8.1f Mpixel/s" % (name, ms, wl.pixels / ms / 1e3), flush=True)
    # kernel level: the backward alone (graph of 12 launches, CUDA events)
    from uemda_b200 import ops
    coef = torch.rand(wl.pixels, device=dev)
    scale = torch.ones(1, device=dev)
    f = lambda s: ops.uvem_loss_backward(s["x1"].detach(), s["x2"].detach(), s["label"], coef, scale)  # noqa: E731
    for s in sets:
        f(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    keep = []
    with torch.cuda.graph(g):
        for i in range(12):
            keep.append(f(sets[i % 3]))
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    print("%-44s %8.1f us" % ("backward, per-block + gather", e0.elapsed_time(e1) * 1e3 / 60), flush=True)


if __name__ == "__main__":
    main()
