"""Speed of the colour JPEG encoder (jpegEncodeColorBatch, degradeJPEGColor) on one GPU, with the card's name, power limit
and max SM clock read in the same run.  Writes one JSON record.

  * batch encode of device-resident 1080p frames into a device blob: 4:2:0 at q50 / q80 / q95 and 4:4:4 at q80, textured
    (a colour gradient with +-20 of noise) and noise content; frames/s, best of --reps after a warm-up.  The batch cycles
    through 48 distinct frames (3 GB for 480 frames, far beyond L2);
  * degradeJPEGColor round trip of the same device batch into a second device batch: frames/s;
  * single-frame latency of both (one device frame, median of 20);
  * cv2.imencode of the same frames on all host threads, in the same run;
  * tools/pointcloud_batch.py's batched pointcloudTest loop with the textures coded on the device (degradeJPEGColor of the
    render's texture batch in place) against textures coded by cv2.imencode / cv2.imdecode on all host threads and copied
    to the device; the views of the two must be identical.
Every stream and every round-trip frame of the timed runs is compared with cv2.

    python tools/jpeg_color_encode_speed.py [--frames 480] [--reps 3] [--out profiles/r13_jpeg_color_encode.json]
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


def host_encode(pool, imgs, q, sampling):
    return list(pool.map(lambda im: cases.encode(im, q, sampling), imgs))


def host_roundtrip(pool, imgs, q, sampling):
    return list(pool.map(lambda im: cv2.imdecode(cases.encode(im, q, sampling), cv2.IMREAD_COLOR), imgs))


def best_time(fn, reps):
    ts = []
    for _ in range(reps):
        sync(); t0 = time.perf_counter()
        fn()
        sync(); ts.append(time.perf_counter() - t0)
    return min(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=480)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pc-frames", type=int, default=32, help="frames of the pointcloudTest loop batch")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r13_jpeg_color_encode.json"))
    a = ap.parse_args()
    threads = os.cpu_count() or 1
    pool = ThreadPoolExecutor(threads)
    n = a.frames
    rec = {"gpu": pcb.gpu_info(), "size": [H, W], "frames": n, "distinct_frames": DISTINCT, "reps": a.reps,
           "host_threads": threads, "cv2": cv2.__version__, "encode": {}}
    src = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    out = torch.empty_like(src)
    for kind in ("textured", "noise"):
        imgs = sources(kind)
        for i in range(n):
            src[i].copy_(torch.from_numpy(imgs[i % DISTINCT]))
        frames = [imgs[i % DISTINCT] for i in range(n)]
        for sampling, q in CONFIGS:
            want = [bytes(s) for s in host_encode(pool, imgs, q, sampling)]
            need = sum(len(want[i % DISTINCT]) for i in range(n))
            blob = torch.empty(need + (1 << 20), dtype=torch.uint8, device="cuda")
            dsrc = (src.data_ptr(), n, H, W)
            enc = lambda: dmc.jpegEncodeColorBatch(dsrc, q, sampling, blob=(blob.data_ptr(), blob.numel()))   # noqa: E731
            _, offsets = enc()                                                                # warm-up: module, scratch
            t_enc = best_time(enc, a.reps)
            _, offsets = enc()
            b = blob[:int(offsets[-1])].cpu().numpy()
            enc_equal = all(bytes(b[int(offsets[i]):int(offsets[i + 1])]) == want[i % DISTINCT] for i in range(n))
            deg = lambda: dmc.degradeJPEGColor(dsrc, q, sampling, dst=out.data_ptr())         # noqa: E731
            deg()
            t_deg = best_time(deg, a.reps)
            _, nbytes = deg()
            ref = [cv2.imdecode(np.frombuffer(w, np.uint8), cv2.IMREAD_COLOR) for w in want]
            got = out.cpu().numpy()
            deg_equal = all(np.array_equal(got[i], ref[i % DISTINCT]) for i in range(n)) and \
                all(int(nbytes[i]) == len(want[i % DISTINCT]) for i in range(n))
            lat_enc, lat_deg = [], []
            one = (src.data_ptr(), 1, H, W)
            for _ in range(20):
                sync(); t0 = time.perf_counter()
                dmc.jpegEncodeColorBatch(one, q, sampling, blob=(blob.data_ptr(), blob.numel()))
                lat_enc.append(time.perf_counter() - t0)
            for _ in range(20):
                sync(); t0 = time.perf_counter()
                dmc.degradeJPEGColor(one, q, sampling, dst=out.data_ptr())
                lat_deg.append(time.perf_counter() - t0)
            host_encode(pool, frames[:threads], q, sampling)
            hs = []
            for _ in range(a.reps):
                t0 = time.perf_counter(); host_encode(pool, frames, q, sampling); hs.append(time.perf_counter() - t0)
            r = {"mean_stream_bytes": int(np.mean([len(w) for w in want])),
                 "gpu_encode_frames_per_s": n / t_enc, "gpu_degrade_frames_per_s": n / t_deg,
                 "gpu_encode_single_frame_latency_ms": 1e3 * statistics.median(lat_enc),
                 "gpu_degrade_single_frame_latency_ms": 1e3 * statistics.median(lat_deg),
                 "cv2_imencode_all_threads_frames_per_s": n / min(hs),
                 "encode_equal_to_cv2": enc_equal, "degrade_equal_to_cv2": deg_equal}
            r["gpu_encode_over_cv2"] = r["gpu_encode_frames_per_s"] / r["cv2_imencode_all_threads_frames_per_s"]
            rec["encode"]["%s_%s_q%d" % (kind, sampling, q)] = r
            print(kind, sampling, q, json.dumps(r), flush=True)
            del blob
    del src, out
    torch.cuda.empty_cache()

    # the batched pointcloudTest loop: textures coded on the device vs coded on the host and copied up
    m = a.pc_frames
    srcs, tex = pcb.sources(m)
    bp = pcb.BatchPath(srcs["synth_disp_1080p"], tex)
    bp.run()
    tex_dev = torch.from_numpy(tex).cuda()
    loop = {"device_texture_coding": [], "host_texture_coding": []}
    for _ in range(a.reps):
        sync(); t0 = time.perf_counter()
        dmc.degradeJPEGColor((tex_dev.data_ptr(), m, H, W), 80, dst=bp.tex.data_ptr())
        sync(); dev_t = time.perf_counter() - t0
        st = bp.run()
        dev_views = bp.views.cpu().numpy()
        loop["device_texture_coding"].append(dict(st, texture=dev_t))
        sync(); t0 = time.perf_counter()
        bp.tex.copy_(torch.from_numpy(np.stack(host_roundtrip(pool, list(tex), 80, "420"))))
        sync(); host_t = time.perf_counter() - t0
        st = bp.run()
        loop["host_texture_coding"].append(dict(st, texture=host_t))
        views_equal = bool(np.array_equal(bp.views.cpu().numpy(), dev_views))
    pc = {"frames": m, "texture": "4:2:0 q80 colour JPEG round trip of tools/pointcloud_batch.py's textures", "views_equal": views_equal}
    for k, runs in loop.items():
        best = min(runs, key=lambda r: sum(r.values()))
        pc[k] = {"frames_per_s": m / sum(best.values()), "ms_per_frame": {s: 1e3 * v / m for s, v in best.items()}}
    rec["pointcloud_loop"] = pc
    print("pointcloud loop", json.dumps(pc), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
