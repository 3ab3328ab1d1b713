#!/usr/bin/env python
"""Resident target set: uem_tile_gather (TileStore.batch) per D4 code against the pinned host -> device copy it replaces.

Two shapes: cfg2 (8 x 6 x 512^2 out of 512^2 tiles) and the LoveDA training shape (16 x 7 x 512^2 crops of 1024^2 tiles).
The stores are several times larger than the 126 MB L2 and every call draws random tiles (and, for crops, random windows),
so the gather reads HBM.  Each code is timed with CUDA events over replays of a CUDA graph of --calls gathers, each with its
own index set (a Python call per gather would time the host).  Algorithmic bytes: fp32 soft in and out, int32 ids in,
int64 ids out; the share of peak is the byte floor at the measured 6536.7 GB/s copy rate over the time.  The host copy is
torch's copy_ of the same soft (fp32) + sup (int64) batch from pinned memory.
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from uemda_b200 import _lib, config  # noqa: E402
from uemda_b200.store import TileStore  # noqa: E402

PEAK_GBS = 6536.7   # measured device copy rate (B200)

SHAPES = {  # name: (tiles in the store, c, tile H, tile W, n, Ho, Wo)
    "cfg2 8x6x512^2 of 512^2": (160, 6, 512, 512, 8, 512, 512),
    "LoveDA 16x7x512^2 of 1024^2": (48, 7, 1024, 1024, 16, 512, 512),
}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def time_graph(fn, calls, reps):
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(g):
        fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * calls)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=64, help="gathers per graph (each with its own random index set)")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    _lib.load()
    config.strict_asserts = False   # no read-back of the status word: the calls are captured
    name, plim = card()
    print("card: %s, power limit %s" % (name, plim), flush=True)
    g = torch.Generator().manual_seed(2333)
    for shape, (T, c, Hs, Ws, n, Ho, Wo) in SHAPES.items():
        st = TileStore(T, c, Hs, Ws, device=dev)
        st.soft.uniform_()
        st.ids.random_(0, 2 ** 20)
        px = n * Ho * Wo
        nbytes = px * (4 * c + 4) + px * (4 * c + 8)
        store_mb = (st.soft.numel() * 4 + st.ids.numel() * 4) / 1e6
        print("\n%s: store %d tiles = %.0f MB, %.1f MB moved per call (%.1f MiB), floor %.1f us at %.1f GB/s"
              % (shape, T, store_mb, nbytes / 1e6, nbytes / 2 ** 20, nbytes / PEAK_GBS / 1e3, PEAK_GBS), flush=True)
        out = (torch.empty(n, c, Ho, Wo, device=dev), torch.empty(n, 1, Ho, Wo, dtype=torch.int64, device=dev))
        print("%-6s %10s %10s %8s" % ("code", "us/call", "GB/s", "of peak"))
        for code in range(8):
            Hw, Ww = (Wo, Ho) if code & 4 else (Ho, Wo)
            sets = []
            for _ in range(args.calls):
                tiles = torch.randint(0, T, (n,), generator=g)
                y0 = torch.randint(0, Hs - Hw + 1, (n,), generator=g)
                x0 = torch.randint(0, Ws - Ww + 1, (n,), generator=g)
                win = torch.stack([y0, x0, torch.full((n,), code)], 1).to(torch.int32)
                sets.append((tiles.to(dev), win.to(dev)))

            def run():
                for t, w in sets:
                    st.batch(t, w, (Ho, Wo), out=out)

            us = time_graph(run, args.calls, args.reps)
            gbs = nbytes / us / 1e3
            print("%-6d %10.2f %10.1f %8.3f" % (code, us, gbs, gbs / PEAK_GBS), flush=True)
        assert int(st.status.item()) == 0
        # what the resident store replaces: the same batch copied from pinned host memory
        h_soft = torch.rand(n, c, Ho, Wo).pin_memory()
        h_sup = torch.randint(0, 2 ** 20, (n, 1, Ho, Wo), dtype=torch.int64).pin_memory()
        d_soft, d_sup = torch.empty_like(h_soft, device=dev), torch.empty_like(h_sup, device=dev)
        for _ in range(3):
            d_soft.copy_(h_soft, non_blocking=True)
            d_sup.copy_(h_sup, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            d_soft.copy_(h_soft, non_blocking=True)
            d_sup.copy_(h_sup, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / args.reps
        hb = h_soft.numel() * 4 + h_sup.numel() * 8
        print("pinned host -> device copy_ of soft fp32 + sup int64 (%.1f MB): %.1f us/batch, %.1f GB/s"
              % (hb / 1e6, us, hb / us / 1e3), flush=True)
        del st, out, sets, h_soft, h_sup, d_soft, d_sup
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
