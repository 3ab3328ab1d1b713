#!/usr/bin/env python
"""Resident source set: uem_label_gather_u8 (LabelStore.batch with downscale) per D4 code, against the two-launch form it
replaces on the device and the pinned host -> device copy it replaces on the host.

Two shapes: cfg2 (8 x 512^2 out of 512^2 tiles, ISPRS bytes, 6 classes) and the LoveDA training shape (16 x 512^2 crops
of 1024^2 tiles, 7 classes), both with DownscaleLabel(16).  The stores (2016 and 1156 tiles: 0.53 and 1.21 GB) are more
than 4x the 126 MB L2 and every call draws random tiles and windows, so the gather reads HBM.  Each code is timed with CUDA
events over replays of a CUDA graph of --calls batches, each with its own index set.  Forms:
  fused      one launch: labels and their DownscaleLabel cells;
  two-launch the gather with down_out = NULL, then uem_downscale_label_i64 on the written labels;
  host copy  torch's copy_ of the (n,Ho,Wo) int64 labels from pinned memory (what the loader path moves per step).
Algorithmic bytes: 1 B in and 8 B out per pixel plus 8 B per cell (the same for both device forms); the share of peak is
that byte floor at the measured 6536.7 GB/s copy rate over the time.
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
from uemda_b200.gast.alignment import DownscaleLabel  # noqa: E402
from uemda_b200.ops import f32  # noqa: E402
from uemda_b200.store import LabelStore  # noqa: E402

PEAK_GBS = 6536.7   # measured device copy rate (B200)
SCALE = 16

SHAPES = {  # name: (tiles in the store, tile H, tile W, n, Ho, Wo, n_classes, lut, a separate ignore byte or None)
    "cfg2 8x512^2 of 512^2 (ISPRS)": (2016, 512, 512, 8, 512, 512, 6, [-1 if v == 255 else v for v in range(256)], 255),
    "LoveDA 16x512^2 of 1024^2": (1156, 1024, 1024, 16, 512, 512, 7, [v - 1 for v in range(256)], None),
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
    ap.add_argument("--calls", type=int, default=64, help="batches per graph (each with its own random index set)")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    lib = L.load()
    config.strict_asserts = False   # no read-back of the status word: the calls are captured
    name, plim = card()
    print("card: %s, power limit %s" % (name, plim), flush=True)
    g = torch.Generator().manual_seed(2333)
    for shape, (T, Hs, Ws, n, Ho, Wo, C, lut, ignore_byte) in SHAPES.items():
        st = LabelStore(T, Hs, Ws, lut, device=dev)
        st.raw.random_(0, C + 1)         # every class and the ignore label (LoveDA: byte 0; ISPRS: byte C, made 255 below)
        if ignore_byte is not None:
            st.raw[st.raw == C] = ignore_byte
        ds = DownscaleLabel(SCALE, C, -1, 0.75)
        px, cells = n * Ho * Wo, n * (Ho // SCALE) * (Wo // SCALE)
        nbytes = px * (1 + 8) + cells * 8
        print("\n%s: store %d tiles = %.0f MB, DownscaleLabel(%d, %d), %.2f MB moved per call (%.2f MiB), floor %.2f us at %.1f GB/s"
              % (shape, T, st.raw.numel() / 1e6, SCALE, C, nbytes / 1e6, nbytes / 2 ** 20, nbytes / PEAK_GBS / 1e3, PEAK_GBS),
              flush=True)
        label = torch.empty(n, Ho, Wo, dtype=torch.int64, device=dev)
        down = torch.empty(n, 1, Ho // SCALE, Wo // SCALE, dtype=torch.int64, device=dev)
        print("%-6s %14s %8s %16s %8s" % ("code", "fused us/call", "of peak", "two-launch us", "of peak"))
        for code in range(8):
            Hw, Ww = (Wo, Ho) if code & 4 else (Ho, Wo)
            sets = []
            for _ in range(args.calls):
                tiles = torch.randint(0, T, (n,), generator=g)
                y0 = torch.randint(0, Hs - Hw + 1, (n,), generator=g)
                x0 = torch.randint(0, Ws - Ww + 1, (n,), generator=g)
                win = torch.stack([y0, x0, torch.full((n,), code)], 1).to(torch.int32)
                sets.append((tiles.to(dev), win.to(dev)))

            def fused():
                for t, w in sets:
                    st.batch(t, w, (Ho, Wo), downscale=ds, out=(label, down))

            def two_launch():
                for t, w in sets:
                    st.batch(t, w, (Ho, Wo), out=(label, None))
                    L.check(lib.uem_downscale_label_i64(L.ptr(label), n, Ho, Wo, SCALE, C, -1, f32(0.75), L.ptr(down), None,
                                                        L.stream_of(label)))

            us_f = time_graph(fused, args.calls, args.reps)
            us_t = time_graph(two_launch, args.calls, args.reps)
            floor = nbytes / PEAK_GBS / 1e3
            print("%-6d %14.2f %8.3f %16.2f %8.3f" % (code, us_f, floor / us_f, us_t, floor / us_t), flush=True)
        assert int(st.status.item()) == 0
        # what the resident store replaces on the host path: the int64 labels copied from pinned memory
        h_lab = torch.randint(-1, C, (n, Ho, Wo), dtype=torch.int64).pin_memory()
        d_lab = torch.empty_like(h_lab, device=dev)
        for _ in range(3):
            d_lab.copy_(h_lab, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            d_lab.copy_(h_lab, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / args.reps
        hb = h_lab.numel() * 8
        print("pinned host -> device copy_ of the int64 labels (%.1f MB): %.1f us/batch, %.1f GB/s" % (hb / 1e6, us, hb / us / 1e3),
              flush=True)
        del st, label, down, sets, h_lab, d_lab
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
