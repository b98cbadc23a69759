"""Coded depth scored by the views it renders: the view-synthesis rate-distortion sweep (dmc_jpeg_view_rd_sweep) on the GPU,
and how fast it runs.  Writes one JSON record.

RD table: qualities 10, 20, ..., 100, standard and optimised Huffman tables, pointcloudTest's filter
filterDisp8U2Depth32F(75, 575, 2.6, 1, 0, 1, 3, 65), isSub, three cameras (R = I with t = (+-100, 0, 0), and the "rot" view
of tests/test_pointcloud.py), K of main.cpp:132-136.  Sources are uncoded: synth_disp frames at 1080p, and the Kinect 16-bit
crop through depth16U2disp8U and the two-pass fillOcclusion (main.cpp:257-260).  The texture is the disparity map itself
(the "depth map view", main.cpp:345-349).  Per quality: mean bytes per frame, and per camera the mean PSNR of the views
rendered from the coded and from the filtered depth against the view of the uncoded depth.  A sample is recomputed on the
CPU (cv2 + the port) and the record says whether it is equal.

Speed, device-resident 1080p synth_disp frames: frame-qualities per second of the sweep, and of the same work through the
public calls (degradeJPEG -> filterDisp8U2Depth32F -> reprojectXYZ -> projectImagefromXYZ -> fillSmallHole -> frameSSE), the
two alternating call by call; the render's share of the sweep (the time a camera adds, per rendered view, over the sweep's
time); the CPU port on all host threads on a sample.

    python tools/view_rd_sweep.py [--frames 24] [--out profiles/r08_view_rd_sweep.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import depthmapcompression_b200 as dmc                      # noqa: E402
from oracle import oracle_py                                # noqa: E402
from _util import load_png                                  # noqa: E402
from test_pointcloud import VIEWS                           # noqa: E402

QUALITIES = list(range(10, 101, 10))
FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6
CHAIN = (1, 0, 1, 3, 65.0)
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


def gray2bgr(frames):
    return np.ascontiguousarray(np.repeat(frames[..., None], 3, axis=-1))


def rd_rows(r, names):
    rows = []
    for k, q in enumerate(QUALITIES):
        row = {"quality": q, "mean_bytes": round(float(r["bytes"][k].astype(np.float64).mean()), 2)}
        for v, name in enumerate(names):
            row[name] = {"mean_psnr_view_coded": round(float(r["psnr_view_coded"][k, v].mean()), 4),
                         "mean_psnr_view_filtered": round(float(r["psnr_view_filtered"][k, v].mean()), 4)}
        rows.append(row)
    return rows


def cpu_view_rd(port, disp, tex, q, opt, f, cams, K):
    """bytes and per-camera SSE of one frame at one quality on the CPU (cv2 + the port)"""
    def view(depth, R, t):
        return port.fill_small_hole(port.project_image(tex, port.reproject_xyz(depth, f), R, t, K, True, rcp=False)[0])
    sse = lambda a, b: int(((a.astype(np.int64) - b) ** 2).sum())       # noqa: E731
    ok, buf = cv2.imencode(".jpg", disp, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, int(opt)])
    dec = cv2.imdecode(buf, 0)
    dz, fz = port.disp8u2depth32f(dec, FB, AMP, 0.0), port.filter_disp8u_depth32f(dec, FOCUS, BASELINE, AMP, *CHAIN)
    out = []
    for R, t in cams:
        ref = view(port.disp8u2depth32f(disp, FB, AMP, 0.0), R, t)
        out.append((sse(ref, view(dz, R, t)), sse(ref, view(fz, R, t))))
    return len(buf), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=24)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_view_rd_sweep.json"))
    args = ap.parse_args()
    params = dmc.filters.chain_params(dmc.capi.CHAIN_DEPTH32F, *CHAIN, focus=FOCUS, baseline=BASELINE, amp=AMP)
    port = oracle_py.Port()
    cams = cameras()
    names = list(cams)
    R = np.stack([c[0] for c in cams.values()]); t = np.stack([c[1] for c in cams.values()])
    modes = {"standard": False, "optimize": True}
    out = {"gpu": gpu_info(), "qualities": QUALITIES, "chain": "filterDisp8U2Depth32F(decoded, 75, 575, 2.6, 1, 0, 1, 3, 65)",
           "coded": "disp8U2depth32F(decoded, 75 * 575, 2.6, 0)", "cameras": {n: {"R": c[0].tolist(), "t": c[1].tolist()} for n, c in cams.items()},
           "view": "fillSmallHole(projectImagefromXYZ(texture, reprojectXYZ(depth, f), R, t, K, isSub=1)), texture = the uncoded disparity as BGR",
           "psnr": "cv::PSNR of the two 8UC3 views from the exact SSE (dmc_psnr_from_sse over 3 * rows * cols)", "rd": {}, "speed": {}}
    print(json.dumps(out["gpu"]), file=sys.stderr, flush=True)

    # ---- RD table ----
    d16 = load_png("kinect_meeting_depth16_crop.png")
    kd = dmc.depth16U2disp8U(d16, None, FB, AMP, 0.0)
    kd = dmc.fillOcclusion(kd, 0, dmc.FILL_DISPARITY)
    kd = np.ascontiguousarray(dmc.fillOcclusion(np.ascontiguousarray(kd.T), 0, dmc.FILL_DISPARITY).T)
    n = args.frames
    synth = np.stack([oracle_py.synth_disp(1080, 1920, 100 + i, shift=(13 * i, 7 * i)) for i in range(n)])
    for name, frames, f in (("kinect_meeting_depth16_crop_filled", kd[None], 510.0), ("synth_disp_1080p", synth, 1100.0)):
        H, W = frames.shape[1:]
        K = intrinsics(f, H, W)
        tex = gray2bgr(frames)
        res = {m: dmc.jpegViewRateDistortion(frames, tex, QUALITIES, params, f, R, t, K, optimize=o, exact_divide=True) for m, o in modes.items()}
        checked, equal = 0, True
        for i in sorted({0, len(frames) - 1}):
            for k, q in enumerate(QUALITIES[::3]):
                kk = QUALITIES.index(q)
                for m, o in modes.items():
                    nb, sse = cpu_view_rd(port, frames[i], tex[i], q, o, f, list(cams.values()), K)
                    got = (int(res[m]["bytes"][kk, i]), [(int(res[m]["sse_view_coded"][kk, v, i]), int(res[m]["sse_view_filtered"][kk, v, i])) for v in range(len(names))])
                    equal &= got == (nb, sse)
                    checked += 1
        out["rd"][name] = {"frames": len(frames), "size": [H, W], "f": f, "cpu_check": {"frame_quality_modes": checked, "equal": bool(equal), "divide": "exact"},
                           **{m: rd_rows(r, names) for m, r in res.items()}}
        print(name, "cpu_check", checked, equal, file=sys.stderr, flush=True)

    # ---- speed: the sweep against the public calls, alternating ----
    H, W = synth.shape[1:]
    f = 1100.0
    K = intrinsics(f, H, W)
    tex = gray2bgr(synth)
    d_src, d_tex = torch.from_numpy(synth).cuda(), torch.from_numpy(tex).cuda()
    torch.cuda.synchronize()
    src, dtex = (d_src.data_ptr(), n, H, W), (d_tex.data_ptr(), n, H, W)
    qs = QUALITIES
    ctx = dmc.default_context()
    pfs = dmc.PostFilterSet()
    d_dec = torch.empty_like(d_src)

    def view(depth, img, Rv, tv):
        return dmc.fillSmallHole(dmc.projectImagefromXYZ(img, None, dmc.reprojectXYZ(depth, None, f), Rv, tv, K, isSub=True))

    def public(o, nq):
        src_h = synth
        ref = [[view(dmc.disp8U2depth32F(src_h[i], None, FB, AMP, 0.0), tex[i], Rv, tv) for Rv, tv in cams.values()] for i in range(n)]
        for q in qs[:nq]:
            dmc.degradeJPEG(src, q, dst=d_dec.data_ptr(), optimize=o)
            ctx.synchronize()
            dec = d_dec.cpu().numpy()
            for i in range(n):
                dz = dmc.disp8U2depth32F(dec[i], None, FB, AMP, 0.0)
                fz = pfs.filterDisp8U2Depth32F(dec[i], None, FOCUS, BASELINE, AMP, *CHAIN)
                for v, (Rv, tv) in enumerate(cams.values()):
                    a = ref[i][v].reshape(1, H, 3 * W)
                    dmc.frameSSE(a, view(dz, tex[i], Rv, tv).reshape(1, H, 3 * W))
                    dmc.frameSSE(a, view(fz, tex[i], Rv, tv).reshape(1, H, 3 * W))

    def sweep(o, nq=len(qs)):
        dmc.jpegViewRateDistortion(src, dtex, qs[:nq], params, f, R, t, K, optimize=o)

    nq_pub = 2                      # the public calls run a subset of the qualities: they take seconds per frame-quality batch
    for m, o in modes.items():
        sweep(o); public(o, 1); torch.cuda.synchronize()                # warm-up
        ts, tp = [], []
        for _ in range(args.reps):
            t0 = time.perf_counter(); sweep(o, nq_pub); ts.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); public(o, nq_pub); tp.append(time.perf_counter() - t0)
        tf = []
        for _ in range(args.reps):
            t0 = time.perf_counter(); sweep(o); tf.append(time.perf_counter() - t0)
        fq, fqf = n * nq_pub, n * len(qs)
        out["speed"][m] = {"sweep_%dq_frame_qualities_per_s" % nq_pub: round(fq / min(ts), 2), "public_calls_%dq_frame_qualities_per_s" % nq_pub: round(fq / min(tp), 2),
                           "speedup_over_public_calls": round(min(tp) / min(ts), 2),
                           "sweep_all_qualities_frame_qualities_per_s": round(fqf / min(tf), 2), "sweep_all_qualities_s": round(min(tf), 3),
                           "sweep_ms_per_frame_quality": round(min(tf) / fqf * 1e3, 3)}
        print(m, json.dumps(out["speed"][m]), file=sys.stderr, flush=True)
    out["speed"]["timing"] = ("wall clock around each call, which returns after its results are on the host; %d device-resident 1080p frames, %d cameras; "
                              "sweep and public calls alternating with %d qualities each (the public calls include the reference views and their "
                              "host round trips, as a user would write them), then the sweep alone over %d qualities; best of %d after a warm-up"
                              % (n, len(names), nq_pub, len(qs), args.reps))

    # ---- the render's share of the sweep: the same sweep with the cameras' renders against with one camera ----
    e = {}
    for nv in (1, len(names)):
        sweep_nv = lambda: dmc.jpegViewRateDistortion(src, dtex, qs, params, f, R[:nv], t[:nv], K)     # noqa: E731
        sweep_nv(); times = []
        for _ in range(args.reps):
            t0 = time.perf_counter(); sweep_nv(); times.append(time.perf_counter() - t0)
        e[nv] = min(times)
    renders_per_camera = n * (1 + 2 * len(qs))
    per_render = (e[len(names)] - e[1]) / ((len(names) - 1) * renders_per_camera)
    total_renders = renders_per_camera * len(names)
    out["speed"]["render_share"] = {"sweep_s_1_camera": round(e[1], 3), "sweep_s_%d_cameras" % len(names): round(e[len(names)], 3),
                                    "ms_per_frame_view": round(per_render * 1e3, 3), "render_share_of_sweep": round(per_render * total_renders / e[len(names)], 3),
                                    "how": "standard tables; the time one more camera adds, per rendered frame view (render, fill, SSE), times the sweep's renders, "
                                           "over the sweep's time"}
    print("render", json.dumps(out["speed"]["render_share"]), file=sys.stderr, flush=True)

    # ---- the CPU port on all host threads, on a sample ----
    cores = os.cpu_count() or 1
    cam_list = list(cams.values())

    def cpu_work(j):
        port.set_num_threads(1)
        cpu_view_rd(port, synth[j % n], tex[j % n], qs[j % len(qs)], False, f, cam_list, K)

    jobs = max(cores, 8)
    with ThreadPoolExecutor(cores) as ex:
        t0 = time.perf_counter(); list(ex.map(cpu_work, range(jobs))); wall = time.perf_counter() - t0
    out["speed"]["cpu"] = {"frame_qualities_per_s": round(jobs / wall, 3), "host_threads": cores, "sample_frame_qualities": jobs,
                           "what": "cv2 encode + decode, the port's converter and filter, %d cameras x (reference, coded, filtered) views rendered and "
                                   "filled by the port, numpy SSE; one 1080p frame-quality per thread" % len(cam_list)}
    print("cpu", json.dumps(out["speed"]["cpu"]), file=sys.stderr, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fo:
        json.dump(out, fo, indent=1)
    print(json.dumps(out["speed"]))


if __name__ == "__main__":
    main()
