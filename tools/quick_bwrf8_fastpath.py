#!/usr/bin/env python
"""Range filter alone (8UC1, radius 5, th 10: the chain's last stage) on three inputs, to see what the flat-strip path
of dmc_bwrf8u_h2.cu buys and costs:
    video   the range filter's real input in bench.py: median 5 -> Gaussian 3 -> min-max 3 of frames of its video
    noise   uniform random bytes: no strip passes the flat test, every warp runs the tap loop
    const   a constant frame: every strip passes the flat test
Each input is --frames 1080p frames stacked into one tall image.  Prints ms per launch (CUDA events over --reps launches),
and from a numpy copy of the kernel's test the share of strips that pass and the share of warps that run the tap loop
once the CTA has regrouped its strips (flat strips first; the one warp holding both counts as a tap warp).  A warp costs
about the same on either path for any data, so  (noise - video) / (noise - const)  is the share of warps that take the
flat path, measured from the timings.

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


def _win(x, axis, lo, hi, fn):
    """fn over offsets lo .. hi along axis, BORDER_REPLICATE"""
    n = x.shape[axis]
    p = np.pad(x, [(-lo, hi) if a == axis else (0, 0) for a in range(x.ndim)], mode="edge")
    out = np.take(p, range(0, n), axis=axis)
    for k in range(1, hi - lo + 1):
        out = fn(out, np.take(p, range(k, k + n), axis=axis))
    return out


def flat_strip_model(img, rad, th, R):
    """numpy copy of the kernel's flat-strip test and regrouping: a strip is 2 pixels x R rows, its footprint the words
    the tap loop reads (pixels x - E .. x + E + 1) over rows y - rad .. y + R - 1 + rad, read through BORDER_REPLICATE; it
    passes iff max(F) - min(centres) <= th and max(centres) - min(F) <= th.  A CTA (128 x 4R pixels, 256 strips, 8 warps)
    runs ceil(tap strips / 32) tap warps.  Returns (share of strips that pass, share of warps that run the tap loop)."""
    x = img.astype(np.int16)
    Hh, Ww = x.shape
    E = 6 if rad <= 6 else (8 if rad <= 8 else 10)
    fmin = _win(_win(x, 0, -rad, R - 1 + rad, np.minimum), 1, -E, E + 1, np.minimum)[::R, ::2]
    fmax = _win(_win(x, 0, -rad, R - 1 + rad, np.maximum), 1, -E, E + 1, np.maximum)[::R, ::2]
    cmin = _win(_win(x, 0, 0, R - 1, np.minimum), 1, 0, 1, np.minimum)[::R, ::2]
    cmax = _win(_win(x, 0, 0, R - 1, np.maximum), 1, 0, 1, np.maximum)[::R, ::2]
    flat = (fmax - cmin <= th) & (cmax - fmin <= th)
    ty, tx = -(-flat.shape[0] // 4), -(-flat.shape[1] // 64)
    tiles = np.ones((4 * ty, 64 * tx), bool)           # strips outside the image go with the flat ones
    tiles[:flat.shape[0], :flat.shape[1]] = flat
    ntap = (~tiles).reshape(ty, 4, tx, 64).sum(axis=(1, 3))
    return float(flat.mean()), float(np.ceil(ntap / 32).sum() / (8 * ty * tx))


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
        strips, tap_warps = flat_strip_model(img, RAD, TH, 4)
        res[name] = {"ms": round(ms, 4), "gpx_s": round(n * H * W / ms / 1e6, 1), "predicted_flat_strips": round(strips, 4),
                     "predicted_tap_warps": round(tap_warps, 4)}
    t = {k: res[k]["ms"] for k in inputs}
    if t["noise"] > t["const"]:
        res["measured_flat_share_video"] = round((t["noise"] - t["video"]) / (t["noise"] - t["const"]), 4)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
