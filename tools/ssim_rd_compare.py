"""Structural similarity next to PSNR: what the SSIM kernel costs, what SSIM adds to both rate-distortion sweeps, and the PSNR
and SSIM table of the three arms (no filter, the post filter set, the boundary reconstruction filter).  Writes one JSON record.

Sources, qualities and arms are those of tools/filter_rd_compare.py (profiles/r09_filter_rd_compare.json): the Kinect 16-bit
crop through depth16U2disp8U and the two-pass fillOcclusion, and 1080p synth_disp frames; qualities 10, 20, ..., 100; gray
sweep PostFilterSet()(2, 1, 3, 5, 10); view sweep filterDisp8U2Depth32F(75, 575, 2.6, 1, 0, 1, 3, 65), isSub, three cameras;
BRF 13x13 (1, 1, 1).  The decoded pixels do not depend on the Huffman mode, so the table is the standard mode's, with the
stream sizes of both modes.  Sampled SSIM entries are recomputed in float64 from cv2 + the CPU port (tests/test_ssim_reference.py)
and the record gives the largest difference.

Speed: frameSSIM on 480 device-resident 1080p frame pairs (gray, and 8UC3 views), larger than L2, CUDA events over at least
one second of calls; both sweeps (device-resident 1080p synth_disp frames, all three arms) with and without SSIM, wall clock
around each call (it returns with the results on the host), alternating in this process.

    python tools/ssim_rd_compare.py [--frames 8] [--reps 5] [--out profiles/r11_ssim_rd.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import depthmapcompression_b200 as dmc                      # noqa: E402
from depthmapcompression_b200 import capi                   # noqa: E402
from oracle import oracle_py                                # noqa: E402
from _util import load_png                                  # noqa: E402
from test_pointcloud import VIEWS                           # noqa: E402
from test_ssim_reference import ssim_ref                    # noqa: E402

QUALITIES = list(range(10, 101, 10))
FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6
VIEW_CHAIN = (1, 0, 1, 3, 65.0)
GRAY_CHAIN = (2, 1, 3, 5, 10)
BRF = ((13, 13), 1.0, 1.0, 1.0)
FB = FOCUS * BASELINE
ARMS = (("none", "coded"), ("post_filter_set", "filtered"), ("brf", "brf"))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    name, power, clock, cur = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "sm_clock_at_start": cur}


def cameras():
    rv = dict((n, (R, t)) for n, R, t in VIEWS)["rot"]
    return {"t=(+100,0,0)": (np.eye(3), np.array([100., 0., 0.])), "t=(-100,0,0)": (np.eye(3), np.array([-100., 0., 0.])), "rot": rv}


def intrinsics(f, H, W):
    K = np.eye(3) * f; K[0, 2] = (W - 1) * 0.5; K[1, 2] = (H - 1) * 0.5; K[2, 2] = 1.0
    return K


def mean(a, nd=4):
    return round(float(np.asarray(a, np.float64).mean()), nd)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_ssim_rd.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    port = oracle_py.Port()
    port.set_num_threads(0)
    pg = dmc.filters.chain_params(capi.CHAIN_DISP8U, *GRAY_CHAIN)
    pv = dmc.filters.chain_params(capi.CHAIN_DEPTH32F, *VIEW_CHAIN, focus=FOCUS, baseline=BASELINE, amp=AMP)
    b = dmc.brf_params(*BRF)
    cams = cameras(); names = list(cams)
    R = np.stack([c[0] for c in cams.values()]); t = np.stack([c[1] for c in cams.values()])
    out = {"gpu": gpu_info(), "qualities": QUALITIES, "brf": "boundaryReconstructionFilter(decoded, Size(13, 13), 1, 1, 1)",
           "gray_chain": "PostFilterSet()(decoded, 2, 1, 3, 5, 10)", "view_chain": "filterDisp8U2Depth32F(decoded, 75, 575, 2.6, 1, 0, 1, 3, 65)",
           "view": "fillSmallHole(projectImagefromXYZ(texture, reprojectXYZ(depth, f), R, t, K, isSub=1)), texture = the uncoded disparity as BGR; "
                   "no filter / BRF depth = disp8U2depth32F(x, 75 * 575, 2.6, 0)",
           "ssim": "mean SSIM, 11x11 Gaussian window sigma 1.5, valid window positions, C1 = (0.01*255)^2, C2 = (0.03*255)^2, views: mean of the "
                   "B, G, R channels (dmc_ssim_batch)", "cameras": names, "rd": {}, "speed": {}}
    print(json.dumps(out["gpu"]), file=sys.stderr, flush=True)

    # ---- PSNR and SSIM of the three arms ----
    d16 = load_png("kinect_meeting_depth16_crop.png")
    kd = dmc.fillOcclusion(dmc.depth16U2disp8U(d16, None, FB, AMP, 0.0), 0, dmc.FILL_DISPARITY)
    kd = np.ascontiguousarray(dmc.fillOcclusion(np.ascontiguousarray(kd.T), 0, dmc.FILL_DISPARITY).T)
    n = args.frames
    synth = np.stack([oracle_py.synth_disp(1080, 1920, 100 + i, shift=(13 * i, 7 * i)) for i in range(n)])
    for name, frames, f, samples in (("kinect_meeting_depth16_crop_filled", kd[None], 510.0, QUALITIES[::3]), ("synth_disp_1080p", synth, 1100.0, (10, 70))):
        H, W = frames.shape[1:]
        K = intrinsics(f, H, W)
        tex = np.ascontiguousarray(np.repeat(frames[..., None], 3, axis=-1))
        g = dmc.jpegRateDistortion(frames, QUALITIES, pg, brf=b, ssim=True)
        v = dmc.jpegViewRateDistortion(frames, tex, QUALITIES, pv, f, R, t, K, exact_divide=True, brf=b, ssim=True)
        gopt = dmc.jpegRateDistortion(frames, QUALITIES, None, optimize=True)
        rows = []
        for k, q in enumerate(QUALITIES):
            row = {"quality": q, "mean_bytes": mean(g["bytes"][k], 2), "mean_bytes_optimize": mean(gopt["bytes"][k], 2),
                   "gray_psnr": {a: mean(g["psnr_" + s][k]) for a, s in ARMS}, "gray_ssim": {a: mean(g["ssim_" + s][k], 6) for a, s in ARMS}}
            for vi, cn in enumerate(names):
                row["view_psnr " + cn] = {a: mean(v["psnr_view_" + s][k, vi]) for a, s in ARMS}
                row["view_ssim " + cn] = {a: mean(v["ssim_view_" + s][k, vi], 6) for a, s in ARMS}
            rows.append(row)
        rec = {"frames": len(frames), "size": [H, W], "f": f, "table": rows}
        # sampled entries against the float64 reference on cv2 + the port: the first frame
        worst, checked = 0.0, 0
        for q in samples:
            k = QUALITIES.index(q)
            dec = cv2.imdecode(cv2.imencode(".jpg", frames[0], [cv2.IMWRITE_JPEG_QUALITY, q])[1], 0)
            bb = port.brf(dec, 13, 13, 1.0, 1.0, 1.0)
            for s, x in (("coded", dec), ("filtered", port.post_filter_set(dec, *GRAY_CHAIN)), ("brf", bb)):
                worst = max(worst, abs(g["ssim_" + s][k, 0] - ssim_ref(frames[0], x))); checked += 1

            def view(depth, Rv, tv):
                return port.fill_small_hole(port.project_image(tex[0], port.reproject_xyz(depth, f), Rv, tv, K, True, rcp=False)[0])
            zs = {"coded": port.disp8u2depth32f(dec, FB, AMP, 0.0), "brf": port.disp8u2depth32f(bb, FB, AMP, 0.0),
                  "filtered": port.filter_disp8u_depth32f(dec, FOCUS, BASELINE, AMP, *VIEW_CHAIN)}
            for vi, (Rv, tv) in enumerate(cams.values()):
                ref = view(port.disp8u2depth32f(frames[0], FB, AMP, 0.0), Rv, tv)
                for s, z in zs.items():
                    worst = max(worst, abs(v["ssim_view_" + s][k, vi, 0] - ssim_ref(ref, view(z, Rv, tv)))); checked += 1
        rec["cpu_check"] = {"values": checked, "max_abs_diff": worst, "what": "SSIM of every arm, gray and every camera's view, frame 0 at q %s, "
                            "against the float64 reference on cv2 + the CPU port; exact division" % list(samples)}
        out["rd"][name] = rec
        print(name, "cpu_check", checked, worst, file=sys.stderr, flush=True)

    # ---- SSIM kernel time: 480 1080p pairs, gray and 8UC3 ----
    ctx = dmc.default_context()
    stream = torch.cuda.Stream(); ctx.set_stream(stream.cuda_stream)
    gen = torch.Generator(device="cuda"); gen.manual_seed(7)
    nb, H, W = 480, 1080, 1920
    for what, cn in (("gray_1080p", 1), ("view_8uc3_1080p", 3)):
        shape = (nb, H, W) if cn == 1 else (nb, H, W, 3)
        da = torch.randint(0, 256, shape, dtype=torch.uint8, device="cuda", generator=gen)
        db = torch.clamp(da.to(torch.int16) + torch.randint(-20, 21, shape, dtype=torch.int16, device="cuda", generator=gen), 0, 255).to(torch.uint8)
        torch.cuda.synchronize()

        def call():
            return dmc.frameSSIM((da.data_ptr(), nb, H, W), (db.data_ptr(), nb, H, W), channels=cn)
        first = call(); call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); call(); e1.record(stream); torch.cuda.synchronize()
        reps = max(2, math.ceil(1000.0 / e0.elapsed_time(e1)))
        e0.record(stream)
        for _ in range(reps):
            last = call()
        e1.record(stream); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        out["speed"]["ssim_" + what] = {"ms_per_frame": round(ms / (reps * nb), 5), "calls": reps, "frames_per_call": nb, "total_ms": round(ms, 1),
                                        "bytes_per_call_mb": round(2 * da.numel() / 2 ** 20, 1), "deterministic": bool(np.array_equal(first, last))}
        print(what, json.dumps(out["speed"]["ssim_" + what]), file=sys.stderr, flush=True)
        del da, db
    out["speed"]["ssim_timing"] = ("CUDA events on the context's stream around back-to-back frameSSIM calls on device tuples (each ends with its "
                                   "results on the host), at least 1 s of calls; inputs larger than L2")

    # ---- both sweeps with and without SSIM, alternating ----
    H, W = synth.shape[1:]
    f = 1100.0
    K = intrinsics(f, H, W)
    tex = np.ascontiguousarray(np.repeat(synth[..., None], 3, axis=-1))
    d_src, d_tex = torch.from_numpy(synth).cuda(), torch.from_numpy(tex).cuda()
    torch.cuda.synchronize()
    src, dtex = (d_src.data_ptr(), n, H, W), (d_tex.data_ptr(), n, H, W)
    fq = n * len(QUALITIES)
    sweeps = {"gray": lambda s: dmc.jpegRateDistortion(src, QUALITIES, pg, brf=b, ssim=s),
              "view": lambda s: dmc.jpegViewRateDistortion(src, dtex, QUALITIES, pv, f, R, t, K, brf=b, ssim=s)}
    for what, fn in sweeps.items():
        fn(False); fn(True)
        ts = {False: [], True: []}
        same = True
        for _ in range(args.reps):
            for s in (False, True):
                t0 = time.perf_counter(); r = fn(s); ts[s].append(time.perf_counter() - t0)
                if s:
                    same &= all(np.array_equal(r[key], r0[key]) for key in r0)
                else:
                    r0 = r
        rec = {"without_ssim_s": {"min": round(min(ts[False]), 4), "median": round(float(np.median(ts[False])), 4)},
               "with_ssim_s": {"min": round(min(ts[True]), 4), "median": round(float(np.median(ts[True])), 4)},
               "ssim_ms_per_frame_quality": round((np.median(ts[True]) - np.median(ts[False])) / fq * 1e3, 4),
               "bytes_and_sse_unchanged": bool(same)}
        out["speed"][what + "_sweep"] = rec
        print(what, json.dumps(rec), file=sys.stderr, flush=True)
    out["speed"]["sweep_timing"] = ("%d device-resident 1080p synth_disp frames, %d qualities, all three arms, %d cameras for the views, standard "
                                    "Huffman tables; wall clock per call, %d calls each, with and without SSIM alternating" % (n, len(QUALITIES), len(names), args.reps))
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fo:
        json.dump(out, fo, indent=1)
    print(json.dumps(out["speed"]))


if __name__ == "__main__":
    main()
