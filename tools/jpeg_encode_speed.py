"""Speed of the GPU JPEG encoder (SURVEY.md 8f-5) on 1080p frames: batch encode, single-frame latency and the degradeJPEG
round trip (encode + decode on the device), next to cv2.imencode on every host thread, timed in the same run.  Clean
(synth_disp), degrade_blocks and uniform-noise frames at q50 / q80 / q95.  Writes one JSON record.

    python tools/jpeg_encode_speed.py [--frames 480] [--out profiles/r04_jpeg_encode.json]
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
import depthmapcompression_b200 as dmc                      # noqa: E402
from oracle.oracle_py import synth_disp, degrade_blocks     # noqa: E402

H, W = 1080, 1920


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:      # the record is still useful without it
        return "%s (nvidia-smi: %s)" % (torch.cuda.get_device_name(0), e)


def timed(fn, reps):
    fn(); torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
    return min(ts), float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=480)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_jpeg_encode.json"))
    args = ap.parse_args()
    n = args.frames
    rs = np.random.RandomState(1)
    clean = [synth_disp(H, W, 1000 + f, shift=(2 * f, f)) for f in range(8)]
    kinds = {"clean": clean, "degrade_blocks": [degrade_blocks(c, i) for i, c in enumerate(clean)],
             "noise": [rs.randint(0, 256, (H, W)).astype(np.uint8) for _ in range(8)]}
    threads = os.cpu_count() or 1
    pool = ThreadPoolExecutor(threads)
    out = {"gpu": gpu_info(), "frame": [H, W], "frames_per_batch": n, "host_threads": threads,
           "timing": "wall clock around each call, which ends in a device synchronise; best and median of 5 calls after a warm-up call; "
                     "device-resident frames and streams", "sets": {}}
    bound = dmc.jpegEncodeBound(H, W)
    for kind, imgs in kinds.items():
        frames = np.stack([imgs[i % 8] for i in range(n)])
        d_src = torch.from_numpy(frames).cuda()
        d_dst = torch.empty_like(d_src)
        for q in (50, 80, 95):
            want = [cv2.imencode(".jpg", imgs[i], [cv2.IMWRITE_JPEG_QUALITY, q])[1].tobytes() for i in range(8)]
            d_blob = torch.empty(n * bound, dtype=torch.uint8, device="cuda")
            # correctness of what is timed
            _, offs = dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), q, blob=(d_blob.data_ptr(), n * bound))
            hb = d_blob[:int(offs[-1])].cpu().numpy()
            assert all(hb[int(offs[i]):int(offs[i + 1])].tobytes() == want[i % 8] for i in range(n)), "%s q%d: stream differs from cv2" % (kind, q)
            best, med = timed(lambda: dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), q, blob=(d_blob.data_ptr(), n * bound)), 5)
            one_best, one_med = timed(lambda: dmc.jpegEncodeGrayBatch((d_src.data_ptr(), 1, H, W), q, blob=(d_blob.data_ptr(), bound)), 20)
            _, nbytes = dmc.degradeJPEG((d_src.data_ptr(), n, H, W), q, dst=d_dst.data_ptr())
            assert [int(x) for x in nbytes] == [len(want[i % 8]) for i in range(n)]
            assert np.array_equal(d_dst[n - 1].cpu().numpy(), cv2.imdecode(np.frombuffer(want[(n - 1) % 8], np.uint8), 0))
            dbest, dmed = timed(lambda: dmc.degradeJPEG((d_src.data_ptr(), n, H, W), q, dst=d_dst.data_ptr()), 5)
            # cv2.imencode on all host threads (OpenCV releases the GIL)
            m = 4 * threads
            enc = lambda i: cv2.imencode(".jpg", imgs[i % 8], [cv2.IMWRITE_JPEG_QUALITY, q])
            list(pool.map(enc, range(threads)))
            t0 = time.perf_counter(); list(pool.map(enc, range(m))); t_cv = time.perf_counter() - t0
            t0 = time.perf_counter(); [enc(i) for i in range(8)]; t_cv1 = (time.perf_counter() - t0) / 8
            res = {"kb_per_frame": round(sum(len(s) for s in want) / 8 / 1e3, 1),
                   "encode_fps": round(n / best), "encode_fps_median": round(n / med),
                   "encode_1_frame_ms": round(one_best * 1e3, 3), "encode_1_frame_ms_median": round(one_med * 1e3, 3),
                   "degrade_roundtrip_fps": round(n / dbest), "degrade_roundtrip_fps_median": round(n / dmed),
                   "cv2_imencode_fps_all_threads": round(m / t_cv), "cv2_imencode_ms_1_thread": round(t_cv1 * 1e3, 2)}
            out["sets"]["%s_q%d" % (kind, q)] = res
            print(kind, q, json.dumps(res), file=sys.stderr, flush=True)
            del d_blob
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
