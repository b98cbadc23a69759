"""The JPEG rate-distortion study of the reference (Fukushima et al., ICME 2013) run on the GPU with dmc_jpeg_rd_sweep, and
how fast it runs.  Writes one JSON record.

RD table: qualities 10, 20, ..., 100, standard and optimised Huffman tables, post filter PostFilterSet()(2, 1, 3, 5, 10), on
the golden frames kinect_meeting_q50, kinect_desk_q50 and x264_depth_y, and on bench.py's video (its x264 frame tiled to
1080p and translated per frame).  Per quality: mean bytes per frame, mean per-frame PSNR of the decoded and of the filtered
frames, and the PSNR of the summed SSE.  These are deterministic; a sample of them is recomputed on the CPU (cv2 + the
port of the chain) and the record says whether they are equal.

Speed, device-resident 1080p frames of the video: frame-qualities per second of the sweep, and of the same work through the
public calls (degradeJPEG -> chain_batch -> frameSSE twice), the two alternating call by call; the SSE kernel alone as bytes
read over CUDA-event time; the CPU path (cv2 encode + decode + the chain, reference build if present, else the port, on all
host threads) on a sample.

    python tools/jpeg_rd_sweep.py [--frames 480] [--out profiles/r06_jpeg_rd_sweep.json]
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
import bench                                                # noqa: E402
import depthmapcompression_b200 as dmc                      # noqa: E402
from oracle import oracle_py                                # noqa: E402
from _util import load_png                                  # noqa: E402

QUALITIES = list(range(10, 101, 10))
CHAIN = (2, 1, 3, 5, 10)
GOLDEN = ("kinect_meeting_q50", "kinect_desk_q50", "x264_depth_y")
HBM_TBS = 7.7               # HGX B200 data sheet, one GPU


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def rd_rows(r, pixels):
    """per quality: mean bytes, mean per-frame PSNR (coded, filtered), PSNR of the summed SSE"""
    n = r["bytes"].shape[1]
    rows = []
    for k, q in enumerate(QUALITIES):
        rows.append({"quality": q, "mean_bytes": round(float(r["bytes"][k].astype(np.float64).mean()), 2),
                     "mean_psnr_coded": round(float(r["psnr_coded"][k].mean()), 4), "mean_psnr_filtered": round(float(r["psnr_filtered"][k].mean()), 4),
                     "psnr_of_summed_sse_coded": round(dmc.psnrFromSSE(int(r["sse_coded"][k].sum()), pixels * n), 4),
                     "psnr_of_summed_sse_filtered": round(dmc.psnrFromSSE(int(r["sse_filtered"][k].sum()), pixels * n), 4)})
    return rows


def cpu_rd(frame, q, optimize, port):
    ok, buf = cv2.imencode(".jpg", frame, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize)])
    assert ok
    dec = cv2.imdecode(buf, 0)
    filt = port.post_filter_set(dec, *CHAIN)
    sse = lambda x: int(((frame.astype(np.int64) - x) ** 2).sum())       # noqa: E731
    return len(buf), sse(dec), sse(filt)


def cpu_check(frames, idx, res, port):
    """the sweep's numbers for frames[idx] against cv2 + the port; -> number of (frame, quality, mode) triples, all equal?"""
    checked, equal = 0, True
    for opt, r in res.items():
        for i in idx:
            for k, q in enumerate(QUALITIES):
                nb, sc, sf = cpu_rd(frames[i], q, opt == "optimize", port)
                equal &= (int(r["bytes"][k, i]), int(r["sse_coded"][k, i]), int(r["sse_filtered"][k, i])) == (nb, sc, sf)
                checked += 1
    return checked, bool(equal)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=480)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_jpeg_rd_sweep.json"))
    args = ap.parse_args()
    params = dmc.filters.chain_params(dmc.capi.CHAIN_DISP8U, *CHAIN)
    port = oracle_py.Port()
    modes = {"standard": False, "optimize": True}
    out = {"gpu": gpu_info(), "qualities": QUALITIES, "chain": "PostFilterSet()(decoded, %d, %d, %d, %d, %d)" % CHAIN,
           "psnr": "cv::PSNR formula from the exact per-frame SSE (dmc_psnr_from_sse)", "rd": {}, "speed": {}}
    print(json.dumps(out["gpu"]), file=sys.stderr, flush=True)

    # ---- RD table ----
    for name in GOLDEN:
        f = load_png(name + ".png")[None]
        res = {m: dmc.jpegRateDistortion(f, QUALITIES, params, optimize=o) for m, o in modes.items()}
        checked, equal = cpu_check(f, [0], res, port)
        out["rd"][name] = {"frames": 1, "size": list(f.shape[1:]), "cpu_check": {"triples": checked, "equal": equal},
                           **{m: rd_rows(r, f[0].size) for m, r in res.items()}}
        print(name, "cpu_check", checked, equal, file=sys.stderr, flush=True)
    base = bench.base_frame()
    H, W = base.shape
    n = args.frames
    video = np.empty((n, H, W), np.uint8)
    for i in range(n):
        video[i] = bench.frame_np(base, i)
    d_src = torch.from_numpy(video).cuda()
    src = (d_src.data_ptr(), n, H, W)
    res = {m: dmc.jpegRateDistortion(src, QUALITIES, params, optimize=o) for m, o in modes.items()}
    sample = [0, n // 3, n - 1]
    checked, equal = cpu_check(video, sample, res, port)
    out["rd"]["bench_video"] = {"frames": n, "size": [H, W], "cpu_check": {"frames": sample, "triples": checked, "equal": equal},
                                **{m: rd_rows(r, H * W) for m, r in res.items()}}
    print("video cpu_check", checked, equal, file=sys.stderr, flush=True)

    # ---- speed: the sweep against the public calls, alternating ----
    ctx = dmc.default_context()
    d_dec, d_filt = torch.empty_like(d_src), torch.empty_like(d_src)

    def public(o):
        for q in QUALITIES:
            dmc.degradeJPEG(src, q, dst=d_dec.data_ptr(), optimize=o)
            ctx.chain_batch(d_dec.data_ptr(), d_filt.data_ptr(), n, H, W, params, device=True)
            dmc.frameSSE(src, (d_dec.data_ptr(), n, H, W)); dmc.frameSSE(src, (d_filt.data_ptr(), n, H, W))
        ctx.synchronize()

    def sweep(o):
        dmc.jpegRateDistortion(src, QUALITIES, params, optimize=o)

    fq = n * len(QUALITIES)
    for m, o in modes.items():
        sweep(o); public(o); torch.cuda.synchronize()           # warm-up
        ts, tp = [], []
        for _ in range(args.reps):
            t0 = time.perf_counter(); sweep(o); ts.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); public(o); tp.append(time.perf_counter() - t0)
        out["speed"][m] = {"sweep_frame_qualities_per_s": round(fq / min(ts)), "sweep_frame_qualities_per_s_median": round(fq / float(np.median(ts))),
                           "public_calls_frame_qualities_per_s": round(fq / min(tp)), "public_calls_frame_qualities_per_s_median": round(fq / float(np.median(tp))),
                           "sweep_us_per_frame_quality": round(min(ts) / fq * 1e6, 2), "public_calls_us_per_frame_quality": round(min(tp) / fq * 1e6, 2)}
        print(m, json.dumps(out["speed"][m]), file=sys.stderr, flush=True)
    out["speed"]["timing"] = ("wall clock around each call, which returns after its results are on the host; %d frame-qualities per call "
                              "(%d device-resident 1080p frames x %d qualities); best and median of %d calls after a warm-up call, the sweep "
                              "and the public calls alternating" % (fq, n, len(QUALITIES), args.reps))

    # ---- speed: the SSE kernel alone ----
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dec = (d_dec.data_ptr(), n, H, W)
    dmc.frameSSE(src, dec)
    times = []
    for _ in range(20):
        e0.record(stream); dmc.frameSSE(src, dec); e1.record(stream); e1.synchronize(); times.append(e0.elapsed_time(e1) / 1e3)
    ctx.set_stream(0)
    read = 2 * n * H * W
    out["speed"]["sse_kernel"] = {"bytes_read": read, "best_s": min(times), "tb_per_s": round(read / min(times) / 1e12, 3),
                                  "tb_per_s_median": round(read / float(np.median(times)) / 1e12, 3), "datasheet_tb_per_s": HBM_TBS,
                                  "timing": "CUDA events on the context's stream around one frameSSE call of two device batches of %d 1080p "
                                            "frames (%.2f GB, larger than L2): output memset + SSE kernel + %d-byte readback; best and median of 20"
                                            % (n, read / 1e9, 8 * n)}
    print("sse", json.dumps(out["speed"]["sse_kernel"]), file=sys.stderr, flush=True)

    # ---- speed: the CPU path on a sample ----
    lib, kind = oracle_py.Port(), "port"
    if oracle_py.Reference.available():
        try:
            lib, kind = oracle_py.Reference(), "reference"
        except Exception:
            pass
    cores = os.cpu_count() or 1

    def cpu_work(j):
        lib.set_num_threads(1)
        f = video[j % 16]
        q = QUALITIES[j % len(QUALITIES)]
        ok, buf = cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, q])
        d = cv2.imdecode(buf, 0)
        lib.post_filter_set(d, *CHAIN)
        return int(((f.astype(np.int32) - d) ** 2).sum())

    jobs = max(2 * cores, 32)
    with ThreadPoolExecutor(cores) as ex:
        list(ex.map(cpu_work, range(cores)))
        t0 = time.perf_counter(); list(ex.map(cpu_work, range(jobs))); wall = time.perf_counter() - t0
    out["speed"]["cpu"] = {"frame_qualities_per_s": round(jobs / wall, 2), "chain": kind, "host_threads": cores, "sample_frame_qualities": jobs,
                           "seconds_for_1000_frames_x_8_qualities": round(8000 / (jobs / wall), 1),
                           "what": "cv2.imencode + cv2.imdecode + the chain + the SSE in numpy per 1080p frame-quality, one per thread"}
    print("cpu", json.dumps(out["speed"]["cpu"]), file=sys.stderr, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["speed"]))


if __name__ == "__main__":
    main()
