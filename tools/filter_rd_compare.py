"""The paper's comparison on the GPU: no filter, the post filter set and the boundary reconstruction filter (BRF) side by side
in both rate-distortion sweeps (dmc_jpeg_rd_sweep_ex, dmc_jpeg_view_rd_sweep_ex), and what the BRF arm costs.  Writes one
JSON record.

RD tables: qualities 10, 20, ..., 100, standard and optimised Huffman tables, BRF 13x13 (1, 1, 1) as pointcloudTest keeps it
(main.cpp:306-311).  Gray sweep: the post filter set PostFilterSet()(2, 1, 3, 5, 10).  View sweep: pointcloudTest's
filterDisp8U2Depth32F(75, 575, 2.6, 1, 0, 1, 3, 65), isSub, three cameras and K as tools/view_rd_sweep.py.  Sources: the
Kinect 16-bit crop through depth16U2disp8U and the two-pass fillOcclusion, and 1080p synth_disp frames.  Sampled entries are
recomputed with cv2 + the CPU port and the record says whether they are equal.

Speed (device-resident 1080p synth_disp frames, best of --reps wall-clock calls that end with the results on the host):
both sweeps with and without the BRF arm; dmc_brf_batch on 480 frames against a loop of dmc_boundary_reconstruction (CUDA
events); with --parent-lib, the single-image BRF and the fused min-max (r = 3) -> BRF of that library and of this build,
alternating (tools/quick_brf.py's case: the Kinect fixture tiled to 1080p, 8-bit, 13x13).

    python tools/filter_rd_compare.py [--frames 8] [--parent-lib path/to/libdmc_b200.so] [--out profiles/r09_filter_rd_compare.json]
"""
import argparse
import ctypes as C
import json
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

QUALITIES = list(range(10, 101, 10))
FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6
VIEW_CHAIN = (1, 0, 1, 3, 65.0)
GRAY_CHAIN = (2, 1, 3, 5, 10)
BRF = ((13, 13), 1.0, 1.0, 1.0)
FB = FOCUS * BASELINE


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def cameras():
    rv = dict((n, (R, t)) for n, R, t in VIEWS)["rot"]
    return {"t=(+100,0,0)": (np.eye(3), np.array([100., 0., 0.])), "t=(-100,0,0)": (np.eye(3), np.array([-100., 0., 0.])), "rot": rv}


def intrinsics(f, H, W):
    K = np.eye(3) * f; K[0, 2] = (W - 1) * 0.5; K[1, 2] = (H - 1) * 0.5; K[2, 2] = 1.0
    return K


def mean(a):
    return round(float(np.asarray(a, np.float64).mean()), 4)


def best(fn, reps):
    fn(); ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return min(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_filter_rd_compare.json"))
    args = ap.parse_args()
    port = oracle_py.Port()
    port.set_num_threads(0)
    pg = dmc.filters.chain_params(capi.CHAIN_DISP8U, *GRAY_CHAIN)
    pv = dmc.filters.chain_params(capi.CHAIN_DEPTH32F, *VIEW_CHAIN, focus=FOCUS, baseline=BASELINE, amp=AMP)
    b = dmc.brf_params(*BRF)
    cams = cameras(); names = list(cams)
    R = np.stack([c[0] for c in cams.values()]); t = np.stack([c[1] for c in cams.values()])
    modes = {"standard": False, "optimize": True}
    out = {"gpu": gpu_info(), "qualities": QUALITIES, "brf": "boundaryReconstructionFilter(decoded, Size(13, 13), 1, 1, 1)",
           "gray_chain": "PostFilterSet()(decoded, 2, 1, 3, 5, 10)", "view_chain": "filterDisp8U2Depth32F(decoded, 75, 575, 2.6, 1, 0, 1, 3, 65)",
           "view": "fillSmallHole(projectImagefromXYZ(texture, reprojectXYZ(depth, f), R, t, K, isSub=1)), texture = the uncoded disparity as BGR; "
                   "no filter / BRF depth = disp8U2depth32F(x, 75 * 575, 2.6, 0)", "cameras": names, "rd": {}, "speed": {}}
    print(json.dumps(out["gpu"]), file=sys.stderr, flush=True)

    # ---- RD tables ----
    d16 = load_png("kinect_meeting_depth16_crop.png")
    kd = dmc.fillOcclusion(dmc.depth16U2disp8U(d16, None, FB, AMP, 0.0), 0, dmc.FILL_DISPARITY)
    kd = np.ascontiguousarray(dmc.fillOcclusion(np.ascontiguousarray(kd.T), 0, dmc.FILL_DISPARITY).T)
    n = args.frames
    synth = np.stack([oracle_py.synth_disp(1080, 1920, 100 + i, shift=(13 * i, 7 * i)) for i in range(n)])
    for name, frames, f in (("kinect_meeting_depth16_crop_filled", kd[None], 510.0), ("synth_disp_1080p", synth, 1100.0)):
        H, W = frames.shape[1:]
        K = intrinsics(f, H, W)
        tex = np.ascontiguousarray(np.repeat(frames[..., None], 3, axis=-1))
        rec = {"frames": len(frames), "size": [H, W], "f": f}
        checked, equal = 0, True
        for m, o in modes.items():
            g = dmc.jpegRateDistortion(frames, QUALITIES, pg, optimize=o, brf=b)
            v = dmc.jpegViewRateDistortion(frames, tex, QUALITIES, pv, f, R, t, K, optimize=o, exact_divide=True, brf=b)
            rows = []
            for k, q in enumerate(QUALITIES):
                row = {"quality": q, "mean_bytes": mean(g["bytes"][k]),
                       "gray_psnr": {"none": mean(g["psnr_coded"][k]), "post_filter_set": mean(g["psnr_filtered"][k]), "brf": mean(g["psnr_brf"][k])}}
                for vi, cn in enumerate(names):
                    row["view_psnr " + cn] = {"none": mean(v["psnr_view_coded"][k, vi]), "post_filter_set": mean(v["psnr_view_filtered"][k, vi]),
                                              "brf": mean(v["psnr_view_brf"][k, vi])}
                rows.append(row)
            rec[m] = rows
            # sampled entries against cv2 + the port: the first and the last frame at q10, q40, q70, q100
            for i in sorted({0, len(frames) - 1}):
                for q in QUALITIES[::3]:
                    k = QUALITIES.index(q)
                    ok, buf = cv2.imencode(".jpg", frames[i], [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, int(o)])
                    dec = cv2.imdecode(buf, 0)
                    bb = port.brf(dec, 13, 13, 1.0, 1.0, 1.0)
                    sse = lambda a, c: int(((a.astype(np.int64) - c) ** 2).sum())      # noqa: E731
                    equal &= int(g["bytes"][k, i]) == len(buf) and int(g["sse_brf"][k, i]) == sse(frames[i], bb)
                    equal &= int(g["sse_filtered"][k, i]) == sse(frames[i], port.post_filter_set(dec, *GRAY_CHAIN))

                    def view(depth, Rv, tv):
                        return port.fill_small_hole(port.project_image(tex[i], port.reproject_xyz(depth, f), Rv, tv, K, True, rcp=False)[0])
                    for vi, (Rv, tv) in enumerate(cams.values()):
                        ref = view(port.disp8u2depth32f(frames[i], FB, AMP, 0.0), Rv, tv)
                        equal &= int(v["sse_view_brf"][k, vi, i]) == sse(ref, view(port.disp8u2depth32f(bb, FB, AMP, 0.0), Rv, tv))
                    checked += 1
        rec["cpu_check"] = {"frame_quality_modes": checked, "equal": bool(equal), "what": "bytes, gray SSE of the post filter set and of the BRF, "
                            "view SSE of the BRF for every camera; exact division"}
        out["rd"][name] = rec
        print(name, "cpu_check", checked, equal, file=sys.stderr, flush=True)

    # ---- speed of the sweeps with and without the BRF arm ----
    H, W = synth.shape[1:]
    f = 1100.0
    K = intrinsics(f, H, W)
    tex = np.ascontiguousarray(np.repeat(synth[..., None], 3, axis=-1))
    d_src, d_tex = torch.from_numpy(synth).cuda(), torch.from_numpy(tex).cuda()
    torch.cuda.synchronize()
    src, dtex = (d_src.data_ptr(), n, H, W), (d_tex.data_ptr(), n, H, W)
    fq = n * len(QUALITIES)
    for m, o in modes.items():
        tg0 = best(lambda: dmc.jpegRateDistortion(src, QUALITIES, pg, optimize=o), args.reps)
        tg1 = best(lambda: dmc.jpegRateDistortion(src, QUALITIES, pg, optimize=o, brf=b), args.reps)
        tv0 = best(lambda: dmc.jpegViewRateDistortion(src, dtex, QUALITIES, pv, f, R, t, K, optimize=o), args.reps)
        tv1 = best(lambda: dmc.jpegViewRateDistortion(src, dtex, QUALITIES, pv, f, R, t, K, optimize=o, brf=b), args.reps)
        out["speed"][m] = {"gray_sweep_frame_qualities_per_s": round(fq / tg0, 1), "gray_sweep_with_brf_frame_qualities_per_s": round(fq / tg1, 1),
                           "gray_brf_arm_ms_per_frame_quality": round((tg1 - tg0) / fq * 1e3, 4),
                           "view_sweep_frame_qualities_per_s": round(fq / tv0, 2), "view_sweep_with_brf_frame_qualities_per_s": round(fq / tv1, 2),
                           "view_brf_arm_ms_per_frame_quality": round((tv1 - tv0) / fq * 1e3, 4)}
        print(m, json.dumps(out["speed"][m]), file=sys.stderr, flush=True)
    out["speed"]["timing"] = ("%d device-resident 1080p synth_disp frames, %d qualities, %d cameras; wall clock around each call (it returns with "
                              "the results on the host), best of %d after a warm-up" % (n, len(QUALITIES), len(names), args.reps))
    del d_src, d_tex

    # ---- dmc_brf_batch against a loop of dmc_boundary_reconstruction: 480 device frames, 1080p, 8-bit, 13x13 ----
    ctx = dmc.default_context()
    stream = torch.cuda.Stream(); ctx.set_stream(stream.cuda_stream)
    img = load_png("kinect_desk_q50.png")
    kin = np.ascontiguousarray(np.tile(img, (3, 3))[:1080, :1920])
    nb = 480
    d_in = torch.from_numpy(np.stack([np.roll(kin, 5 * i, axis=1) for i in range(nb)])).cuda()
    d_out, d_loop = torch.empty_like(d_in), torch.empty_like(d_in)
    torch.cuda.synchronize()
    fpx = 1080 * 1920
    imgs = [(capi.DmcImage(d_in.data_ptr() + i * fpx, 1080, 1920, 0, 0, 1), capi.DmcImage(d_loop.data_ptr() + i * fpx, 1080, 1920, 0, 0, 1)) for i in range(nb)]

    def batch():
        dmc.boundaryReconstructionFilterBatch((d_in.data_ptr(), nb, 1080, 1920), d_out.data_ptr(), *BRF)

    def loop():
        for s_, d_ in imgs:
            ctx.check(capi.lib.dmc_boundary_reconstruction(ctx.h, C.byref(s_), C.byref(d_), 13, 13, 1.0, 1.0, 1.0))

    def ev_ms(fn, reps):
        fn(); torch.cuda.synchronize(); r = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); fn(); e1.record(stream); torch.cuda.synchronize(); r.append(e0.elapsed_time(e1))
        return min(r)

    tb, tl = [], []
    for _ in range(args.reps):
        tb.append(ev_ms(batch, 1)); tl.append(ev_ms(loop, 1))
    out["speed"]["brf_batch_480x1080p_u8_13x13"] = {"batch_ms": round(min(tb), 3), "loop_ms": round(min(tl), 3), "batch_ms_per_frame": round(min(tb) / nb, 4),
                                                    "loop_ms_per_frame": round(min(tl) / nb, 4), "equal": bool(torch.equal(d_out, d_loop)),
                                                    "timing": "CUDA events on the context's stream, best of %d, batch and loop alternating" % args.reps}
    print("brf batch", json.dumps(out["speed"]["brf_batch_480x1080p_u8_13x13"]), file=sys.stderr, flush=True)
    del d_in, d_out, d_loop

    # ---- single-image BRF and fused min-max -> BRF: the parent library and this build, alternating ----
    if args.parent_lib:
        parent = C.CDLL(os.path.abspath(args.parent_lib))
        IMG = C.POINTER(capi.DmcImage)
        parent.dmc_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        parent.dmc_destroy.argtypes = [C.c_void_p]; parent.dmc_destroy.restype = None
        parent.dmc_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        parent.dmc_boundary_reconstruction.argtypes = [C.c_void_p, IMG, IMG, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float]
        parent.dmc_minmax_boundary_reconstruction.argtypes = [C.c_void_p, IMG, IMG, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float]
        libs = {"parent": parent, "this": capi.lib}                 # (capi.lib carries its own signatures)
        s1 = torch.from_numpy(kin).cuda(); o1 = torch.empty_like(s1); o2 = torch.empty_like(s1); torch.cuda.synchronize()
        si, oi = capi.DmcImage(s1.data_ptr(), 1080, 1920, 0, 0, 1), capi.DmcImage(o1.data_ptr(), 1080, 1920, 0, 0, 1)
        ctxs = {}
        for k, lib in libs.items():
            h = C.c_void_p(); assert lib.dmc_create(0, C.byref(h)) == 0
            assert lib.dmc_set_stream(h, C.c_void_p(stream.cuda_stream)) == 0
            ctxs[k] = h
        calls = {"single_image_brf_kinect_1080p_u8_13x13": lambda k: libs[k].dmc_boundary_reconstruction(ctxs[k], C.byref(si), C.byref(oi), 13, 13, 1.0, 1.0, 1.0),
                 "fused_minmax3_brf_kinect_1080p_u8_13x13": lambda k: libs[k].dmc_minmax_boundary_reconstruction(ctxs[k], C.byref(si), C.byref(oi), 3, 13, 13, 1.0, 1.0, 1.0)}
        for what, call in calls.items():
            res = {k: [] for k in libs}

            def one(k, reps=50):
                for _ in range(reps):
                    assert call(k) == 0
            for k in libs:
                one(k, 5)
            for _ in range(7):
                for k in libs:
                    res[k].append(ev_ms(lambda: one(k), 1) / 50)
            one("parent", 1); torch.cuda.synchronize(); o2.copy_(o1); one("this", 1); torch.cuda.synchronize()
            rec = {k: {"min_ms": round(min(v), 4), "median_ms": round(float(np.median(v)), 4)} for k, v in res.items()}
            rec["equal"] = bool(torch.equal(o1, o2))
            rec["timing"] = "CUDA events, 50 device-resident calls per sample, 7 samples per library, alternating; Kinect fixture tiled to 1080p"
            out["speed"][what] = rec
            print(what, json.dumps(rec), file=sys.stderr, flush=True)
        torch.cuda.synchronize()
        for k, lib in libs.items():
            lib.dmc_destroy(ctxs[k])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fo:
        json.dump(out, fo, indent=1)
    print(json.dumps(out["speed"]))


if __name__ == "__main__":
    main()
