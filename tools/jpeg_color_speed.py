"""Speed of the colour JPEG decoder (jpegDecodeColorBatch) on one GPU, with the card's name, power limit and max SM clock
read in the same run.  Writes one JSON record.

  * batch decode of 1080p frames from a host blob to device memory: 4:2:0 at q50 / q80 / q95 and 4:4:4 at q80, textured
    (a colour gradient with +-20 of noise) and noise content; frames/s, best of --reps after a warm-up.  The batch cycles
    through 48 distinct frames, so the blob (about 80-800 MB) does not stay in L2;
  * single-frame latency (one stream to device memory, median);
  * cv2.imdecode(IMREAD_COLOR) of the same streams on all host threads, in the same run;
  * tools/pointcloud_batch.py's batched pointcloudTest loop with the textures decoded on the device (jpegDecodeColorBatch
    into the render's texture batch) against textures decoded by cv2 on all host threads and copied to the device.
Every decoded frame of the timed runs is compared with cv2.

    python tools/jpeg_color_speed.py [--frames 480] [--reps 3] [--out profiles/r12_jpeg_color.json]
"""
import argparse
import json
import os
import statistics
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import depthmapcompression_b200 as dmc                      # noqa: E402
import _jpeg_color_cases as cases                           # noqa: E402
import pointcloud_batch as pcb                              # noqa: E402

H, W, DISTINCT = 1080, 1920, 48
CONFIGS = [("420", 50), ("420", 80), ("420", 95), ("444", 80)]


def sync():
    dmc.default_context().synchronize()
    torch.cuda.synchronize()


def sources(kind):
    rs = np.random.RandomState(7)
    if kind == "textured":
        return [cases.textured(H, W, i) for i in range(DISTINCT)]
    return [rs.randint(0, 256, (H, W, 3)).astype(np.uint8) for _ in range(DISTINCT)]


def host_decode(pool, streams):
    return list(pool.map(lambda s: cv2.imdecode(s, cv2.IMREAD_COLOR), streams))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=480)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pc-frames", type=int, default=32, help="frames of the pointcloudTest loop batch")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_jpeg_color.json"))
    a = ap.parse_args()
    threads = os.cpu_count() or 1
    pool = ThreadPoolExecutor(threads)
    rec = {"gpu": pcb.gpu_info(), "size": [H, W], "frames": a.frames, "distinct_frames": DISTINCT, "reps": a.reps,
           "host_threads": threads, "cv2": cv2.__version__, "decode": {}}
    out = torch.empty((a.frames, H, W, 3), dtype=torch.uint8, device="cuda")
    for kind in ("textured", "noise"):
        imgs = sources(kind)
        for sampling, q in CONFIGS:
            enc = [cases.encode(im, q, sampling) for im in imgs]
            streams = [enc[i % DISTINCT] for i in range(a.frames)]
            blob, offsets = dmc.pack_streams(streams)
            dmc.jpegDecodeColorBatch((blob, offsets), H, W, dst=out.data_ptr())          # warm-up: module, scratch
            ts = []
            for _ in range(a.reps):
                sync(); t0 = time.perf_counter()
                dmc.jpegDecodeColorBatch((blob, offsets), H, W, dst=out.data_ptr())
                sync(); ts.append(time.perf_counter() - t0)
            want = host_decode(pool, enc)
            host_decode(pool, streams[:threads])
            hs = []
            for _ in range(a.reps):
                t0 = time.perf_counter(); host_decode(pool, streams); hs.append(time.perf_counter() - t0)
            got = out.cpu().numpy()
            equal = all(np.array_equal(got[i], want[i % DISTINCT]) for i in range(a.frames))
            lat = []
            one = dmc.pack_streams(streams[:1])
            for _ in range(20):
                sync(); t0 = time.perf_counter()
                dmc.jpegDecodeColorBatch(one, H, W, dst=out.data_ptr())
                lat.append(time.perf_counter() - t0)
            r = {"mean_stream_bytes": int(np.mean([s.size for s in enc])), "gpu_frames_per_s": a.frames / min(ts),
                 "gpu_single_frame_latency_ms": 1e3 * statistics.median(lat),
                 "cv2_all_threads_frames_per_s": a.frames / min(hs), "equal_to_cv2": equal}
            r["gpu_over_cv2"] = r["gpu_frames_per_s"] / r["cv2_all_threads_frames_per_s"]
            rec["decode"]["%s_%s_q%d" % (kind, sampling, q)] = r
            print(kind, sampling, q, json.dumps(r), flush=True)

    # the batched pointcloudTest loop: textures decoded on the device vs on the host
    n = a.pc_frames
    srcs, tex = pcb.sources(n)
    d16 = srcs["synth_disp_1080p"]
    tstreams = [cases.encode(t, 80, "420") for t in tex]
    tblob = dmc.pack_streams(tstreams)
    bp = pcb.BatchPath(d16, tex)
    bp.run()
    loop = {"device_texture_decode": [], "host_texture_decode": []}
    for _ in range(a.reps):
        sync(); t0 = time.perf_counter()
        dmc.jpegDecodeColorBatch(tblob, H, W, dst=bp.tex.data_ptr())
        sync(); dev_t = time.perf_counter() - t0
        st = bp.run()
        dev_views = bp.views.cpu().numpy()
        loop["device_texture_decode"].append(dict(st, texture=dev_t))
        sync(); t0 = time.perf_counter()
        bp.tex.copy_(torch.from_numpy(np.stack(host_decode(pool, tstreams))))
        sync(); host_t = time.perf_counter() - t0
        st = bp.run()
        loop["host_texture_decode"].append(dict(st, texture=host_t))
        views_equal = bool(np.array_equal(bp.views.cpu().numpy(), dev_views))
    pc = {"frames": n, "texture": "4:2:0 q80 colour JPEG of tools/pointcloud_batch.py's textures", "views_equal": views_equal}
    for k, runs in loop.items():
        best = min(runs, key=lambda r: sum(r.values()))
        pc[k] = {"frames_per_s": n / sum(best.values()), "ms_per_frame": {s: 1e3 * v / n for s, v in best.items()}}
    rec["pointcloud_loop"] = pc
    print("pointcloud loop", json.dumps(pc), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
