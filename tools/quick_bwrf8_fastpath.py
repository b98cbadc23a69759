#!/usr/bin/env python
"""Range filter alone (8UC1, radius 5, th 10: the chain's last stage) on three inputs, to see what the flat-warp path
of dmc_bwrf8u_h2.cu buys and costs:
    video   the range filter's real input in bench.py: median 5 -> Gaussian 3 -> min-max 3 of frames of its video
    noise   uniform random bytes: no warp passes the flat test, every warp runs the tap loop
    const   a constant frame: every warp passes the flat test
Each input is --frames 1080p frames stacked into one tall image.  Prints ms per launch (CUDA events over --reps launches)
and the share of warps that pass the flat test, as predicted by a numpy copy of the test.  Both paths cost the same
for any data, so  (noise - video) / (noise - const)  is the share of the flat path measured from the timings.

    python tools/quick_bwrf8_fastpath.py [--frames 8] [--reps 50]"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RAD, TH = 5, 10
H, W = 1080, 1920


def flat_warp_share(img, rad, th, R):
    """numpy copy of the kernel's flat-warp test: warps of 32 x 2R pixels in tiles of 128 x 4R; footprint = the warp's
    rows +- rad and the 4-pixel chunks (counted from 16 pixels left of the tile) that hold its columns +- rad, all read
    through BORDER_REPLICATE; the warp passes iff max(F) - min(centres) <= th and max(centres) - min(F) <= th."""
    x = img.astype(np.int16)
    Hh, Ww = x.shape
    q0 = (16 - rad) >> 2
    nq = ((16 + 31 + rad) >> 2) - q0 + 1
    ntx, nty = (Ww + 127) // 128, (Hh + 4 * R - 1) // (4 * R)
    pl, pt = 16, rad
    xp = np.pad(x, ((pt, nty * 4 * R + rad - Hh), (pl, ntx * 128 + 16 - Ww + 8)), mode="edge")      # xp[pt + y, pl + x] = x[clamp(y), clamp(x)]
    passed = total = 0
    for ty in range(nty):
        for wy in range(2):
            y0 = ty * 4 * R + wy * 2 * R
            rows = xp[y0:y0 + 2 * R + 2 * rad]
            cen = xp[pt + y0:pt + y0 + 2 * R]
            for tx in range(ntx):
                for wx in range(4):
                    s0 = tx * 128 + 4 * (8 * wx + q0)          # padded column of the first chunk (staged column - 16 + pl)
                    f = rows[:, s0:s0 + 4 * nq]
                    c = cen[:, pl + tx * 128 + 32 * wx:pl + tx * 128 + 32 * wx + 32]
                    passed += (f.max() - c.min() <= th) and (c.max() - f.min() <= th)
                    total += 1
    return passed / total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    import torch
    import depthmapcompression_b200 as dmc
    from depthmapcompression_b200.capi import DmcImage, lib
    import bench

    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = dmc.Context(0)
    ctx.set_stream(stream.cuda_stream)

    base = bench.base_frame()
    n = args.frames
    video = []
    for i in range(n):
        f = bench.frame_np(base, i * 1000 // n)
        m = dmc.medianBlur(f, None, 5, ctx=ctx)
        g = dmc.smallGaussianBlur(m, None, 3, 1.5, ctx=ctx)
        video.append(dmc.blurRemoveMinMax(g, None, 3, ctx=ctx))
    inputs = {"video": np.concatenate(video), "noise": np.random.RandomState(1).randint(0, 256, (n * H, W)).astype(np.uint8),
              "const": np.full((n * H, W), 128, np.uint8)}
    res = {"gpu": torch.cuda.get_device_name(0), "shape": [n * H, W], "radius": RAD, "th": TH, "reps": args.reps}
    for name, img in inputs.items():
        d_in = torch.from_numpy(img).to(dev)
        d_out = torch.empty_like(d_in)
        s8 = DmcImage(d_in.data_ptr(), n * H, W, 0, 0, 1)
        o8 = DmcImage(d_out.data_ptr(), n * H, W, 0, 0, 1)
        call = lambda: lib.dmc_bwrf(ctx.h, C.byref(s8), C.byref(o8), 2 * RAD + 1, 2 * RAD + 1, float(TH), 0, 1)
        for _ in range(5):
            assert call() == 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(args.reps):
            call()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.reps
        res[name] = {"ms": round(ms, 4), "gpx_s": round(n * H * W / ms / 1e6, 1), "predicted_flat_warps": round(flat_warp_share(img, RAD, TH, 4), 4)}
    t = {k: res[k]["ms"] for k in inputs}
    if t["noise"] > t["const"]:
        res["measured_flat_share_video"] = round((t["noise"] - t["video"]) / (t["noise"] - t["const"]), 4)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
