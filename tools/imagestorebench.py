#!/usr/bin/env python
"""Resident image set: uem_image_gather_u8 (ImageStore.batch) per D4 code, in both store forms, against the same cut written
as device-side torch ops and the pinned host -> device copy of the fp32 batch that it replaces.

Two shapes, C = 3 (RGB / IRRG): cfg2 (8 x 512^2 out of 2016 tiles of 512^2) and the LoveDA training shape (16 x 512^2
crops of 1156 tiles of 1024^2).  The stores (1.59 and 3.64 GB) are far larger than the 126 MB L2 and every call draws
random tiles and windows, so the gather reads HBM.  Each code is timed with CUDA events over replays of a CUDA graph of
--calls batches, each with its own index set.  Forms:
  16-byte   the entry point's 16-byte store form (Wo % 4 == 0, out 16-byte aligned);
  4-byte    its 4-byte store form (out 4 bytes past a 16-byte boundary);
  torch     per sample: index the tile, slice the window, flip, transpose, then table[ch, bytes] (torch's gather kernels);
  host copy torch's copy_ of the (n,C,Ho,Wo) fp32 batch from pinned memory (what the loader path moves per step).
Algorithmic bytes: C B in and 4C B out per pixel; the share of peak is that byte floor at the measured 6536.7 GB/s copy
rate over the time.
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from uemda_b200 import _lib as L  # noqa: E402
from uemda_b200 import config  # noqa: E402
from uemda_b200.store import ImageStore  # noqa: E402

PEAK_GBS = 6536.7   # measured device copy rate (B200)
C = 3
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)

SHAPES = {  # name: (tiles in the store, tile H, tile W, n, Ho, Wo)
    "cfg2 8x512^2 of 512^2": (2016, 512, 512, 8, 512, 512),
    "LoveDA 16x512^2 of 1024^2": (1156, 1024, 1024, 16, 512, 512),
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


def torch_cut(raw, table, tiles, windows, Ho, Wo, out):
    """The cut as device-side torch ops, one sample at a time (the windows are host values, fixed at capture)."""
    ch = torch.arange(C, device=raw.device).view(-1, 1, 1)
    for s, (t, (y0, x0, code)) in enumerate(zip(tiles, windows)):
        Hw, Ww = (Wo, Ho) if code & 4 else (Ho, Wo)
        x = raw[t, y0:y0 + Hw, x0:x0 + Ww].permute(2, 0, 1)
        dims = [d for d, f in ((-2, code & 2), (-1, code & 1)) if f]
        if dims:
            x = x.flip(dims)
        if code & 4:
            x = x.transpose(-2, -1)
        out[s] = table[ch, x.long()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=64, help="batches per graph (each with its own random index set)")
    ap.add_argument("--torch-calls", type=int, default=8, help="batches per graph of the torch form")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    L.load()
    config.strict_asserts = False   # no read-back of the status word: the calls are captured
    name, plim = card()
    print("card: %s, power limit %s" % (name, plim), flush=True)
    g = torch.Generator().manual_seed(2333)
    for shape, (T, Hs, Ws, n, Ho, Wo) in SHAPES.items():
        st = ImageStore(T, Hs, Ws, C, ImageStore.normalize_table(MEAN, STD), device=dev)
        st.raw.random_(0, 256)
        nbytes = n * Ho * Wo * C * (1 + 4)
        floor = nbytes / PEAK_GBS / 1e3
        print("\n%s, C = %d: store %d tiles = %.2f GB, %.2f MB moved per call (%.2f MiB), floor %.2f us at %.1f GB/s"
              % (shape, C, T, st.raw.numel() / 1e9, nbytes / 1e6, nbytes / 2 ** 20, floor, PEAK_GBS), flush=True)
        buf = torch.empty(n * C * Ho * Wo + 4, dtype=torch.float32, device=dev)
        assert buf.data_ptr() % 16 == 0
        out16 = buf[:n * C * Ho * Wo].view(n, C, Ho, Wo)
        out4 = buf[1:1 + n * C * Ho * Wo].view(n, C, Ho, Wo)
        print("%-6s %14s %8s %14s %8s %14s %8s" % ("code", "16-byte us", "of peak", "4-byte us", "of peak", "torch us", "of peak"))
        for code in range(8):
            Hw, Ww = (Wo, Ho) if code & 4 else (Ho, Wo)
            sets = []
            for _ in range(args.calls):
                tiles = torch.randint(0, T, (n,), generator=g)
                y0 = torch.randint(0, Hs - Hw + 1, (n,), generator=g)
                x0 = torch.randint(0, Ws - Ww + 1, (n,), generator=g)
                win = torch.stack([y0, x0, torch.full((n,), code)], 1).to(torch.int32)
                sets.append((tiles.to(dev), win.to(dev), tiles.tolist(), win.tolist()))

            def gather(out):
                def fn():
                    for t, w, _, _ in sets:
                        st.batch(t, w, (Ho, Wo), out=out)
                return fn

            def by_torch():
                for _, _, tl, wl in sets[:args.torch_calls]:
                    torch_cut(st.raw, st.table, tl, wl, Ho, Wo, out16)

            us16 = time_graph(gather(out16), args.calls, args.reps)
            us4 = time_graph(gather(out4), args.calls, args.reps)
            ust = time_graph(by_torch, args.torch_calls, args.reps)
            print("%-6d %14.2f %8.3f %14.2f %8.3f %14.2f %8.3f" % (code, us16, floor / us16, us4, floor / us4, ust, floor / ust),
                  flush=True)
            # the three forms agree on the last batch
            _, _, tl, wl = sets[-1]
            st.batch(sets[-1][0], sets[-1][1], (Ho, Wo), out=out4)
            want = torch.empty_like(out16)
            torch_cut(st.raw, st.table, tl, wl, Ho, Wo, want)
            assert torch.equal(st.batch(tl, wl, (Ho, Wo)), want) and torch.equal(out4, want)
        assert int(st.status.item()) == 0
        # what the resident store replaces on the host path: the fp32 batch copied from pinned memory
        h_img = torch.randn(n, C, Ho, Wo).pin_memory()
        d_img = torch.empty_like(h_img, device=dev)
        for _ in range(3):
            d_img.copy_(h_img, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            d_img.copy_(h_img, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / args.reps
        hb = h_img.numel() * 4
        print("pinned host -> device copy_ of the fp32 batch (%.1f MB): %.1f us/batch, %.1f GB/s" % (hb / 1e6, us, hb / us / 1e3),
              flush=True)
        del st, buf, out16, out4, sets, h_img, d_img
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
