"""Speed and size of the GPU JPEG encoder with optimised Huffman tables next to the standard tables, timed alternately in
one run on 1080p frames: clean (synth_disp), degrade_blocks and uniform-noise frames at q50 / q80 / q95.  Per set: KB per
frame in both modes, encode and degradeJPEG round-trip frames/s in both modes, jpegDecodeGrayBatch frames/s from a host
blob of the optimised (per-frame-table) streams, and cv2.imencode with and without IMWRITE_JPEG_OPTIMIZE on all host
threads.  Also the host parse time of 2048 small per-frame-table streams with the hashed table de-duplication of
csrc/dmc_jpeg_parse.h and with the linear scan it replaced.  Writes one JSON record.

    python tools/jpeg_encode_optimize_speed.py [--frames 480] [--out profiles/r05_jpeg_encode_optimize.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
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

PARSE_BENCH = r"""
#include "dmc_jpeg_parse.h"
#include <chrono>
#include <cstdio>
using namespace dmc;
// the linear first-occurrence scan the hashed pools replaced
template <class T> static int linear(std::vector<T>& pool, const T& v) {
    for (size_t i = 0; i < pool.size(); i++) if (memcmp(&pool[i], &v, sizeof(T)) == 0) return (int)i;
    pool.push_back(v); return (int)pool.size() - 1;
}
int main(int argc, char** argv) {
    FILE* f = fopen(argv[1], "rb"); std::vector<uint8_t> blob; uint8_t b[65536]; size_t k;
    while ((k = fread(b, 1, sizeof b, f)) > 0) blob.insert(blob.end(), b, b + k);
    fclose(f);
    std::vector<uint64_t> off; f = fopen(argv[2], "rb"); uint64_t o; while (fread(&o, 8, 1, f) == 1) off.push_back(o); fclose(f);
    const int n = (int)off.size() - 1;
    double best_h = 1e9, best_l = 1e9; size_t nh = 0, nl = 0;
    for (int rep = 0; rep < 5; rep++) {
        auto t0 = std::chrono::steady_clock::now();
        JpegTablePools pools; FrameDesc d;
        for (int i = 0; i < n; i++) jpeg_parse_frame(blob.data() + off[i], off[i + 1] - off[i], off[i], -1, -1, pools, &d);
        auto t1 = std::chrono::steady_clock::now();
        std::vector<QuantTable> lq; std::vector<HuffTable> lh;
        for (int i = 0; i < n; i++) {
            std::vector<QuantTable> q1; std::vector<HuffTable> h1;
            jpeg_parse_frame(blob.data() + off[i], off[i + 1] - off[i], off[i], -1, -1, q1, h1, &d);
            linear(lq, q1[d.qt]); linear(lh, h1[d.dc]); linear(lh, h1[d.ac]);
        }
        auto t2 = std::chrono::steady_clock::now();
        best_h = std::min(best_h, std::chrono::duration<double>(t1 - t0).count());
        best_l = std::min(best_l, std::chrono::duration<double>(t2 - t1).count());
        nh = pools.h.items.size(); nl = lh.size();
    }
    printf("{\"hashed_ms\": %.3f, \"linear_ms\": %.3f, \"distinct_huffman_tables\": %zu, \"linear_distinct\": %zu}\n", best_h * 1e3, best_l * 1e3, nh, nl);
    return 0;
}
"""


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


def cv2_enc(img, q, opt):
    return cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, int(opt)])[1].tobytes()


def parse_bench():
    """Host parse of 2048 small per-frame-table streams (mixed qualities), hashed vs linear de-duplication (the parser
    header compiled as it is into a stand-alone timing program in a temporary directory)."""
    rs = np.random.RandomState(3)
    base = np.clip(rs.normal(110, 35, (32, 48)), 0, 255).astype(np.uint8)
    streams = []
    for i in range(2048):
        img = base.copy(); img[rs.randint(0, 32, 16), rs.randint(0, 48, 16)] = rs.randint(0, 256, 16)
        streams.append(cv2_enc(img, int(rs.randint(5, 100)), True))
    blob, offsets = dmc.pack_streams(streams)
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "parse_bench.cpp"), os.path.join(d, "parse_bench")
        open(src, "w").write(PARSE_BENCH)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "depthmapcompression_b200", "csrc"), "-o", exe, src])
        blob[:int(offsets[-1])].tofile(os.path.join(d, "blob")); offsets.astype(np.uint64).tofile(os.path.join(d, "offs"))
        r = json.loads(subprocess.check_output([exe, os.path.join(d, "blob"), os.path.join(d, "offs")], text=True))
    r["streams"] = len(streams)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=480)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_jpeg_encode_optimize.json"))
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
                     "device-resident frames and streams for encode and degrade, the two modes alternating call by call; "
                     "decode from a host blob of the optimised streams", "sets": {}}
    out["parse_2048_per_frame_table_streams"] = parse_bench()
    print("parse", json.dumps(out["parse_2048_per_frame_table_streams"]), file=sys.stderr, flush=True)
    modes = {"standard": False, "optimize": True}
    for kind, imgs in kinds.items():
        frames = np.stack([imgs[i % 8] for i in range(n)])
        d_src = torch.from_numpy(frames).cuda()
        d_dst = torch.empty_like(d_src)
        for q in (50, 80, 95):
            bound = dmc.jpegEncodeBound(H, W, optimize=True)
            d_blob = torch.empty(n * bound, dtype=torch.uint8, device="cuda")
            res = {}
            want = {m: [cv2_enc(imgs[i], q, o) for i in range(8)] for m, o in modes.items()}
            for m, o in modes.items():           # correctness of what is timed
                _, offs = dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), q, blob=(d_blob.data_ptr(), n * bound), optimize=o)
                hb = d_blob[:int(offs[-1])].cpu().numpy()
                assert all(hb[int(offs[i]):int(offs[i + 1])].tobytes() == want[m][i % 8] for i in range(n)), "%s q%d %s: stream differs from cv2" % (kind, q, m)
                _, nbytes = dmc.degradeJPEG((d_src.data_ptr(), n, H, W), q, dst=d_dst.data_ptr(), optimize=o)
                assert [int(x) for x in nbytes] == [len(want[m][i % 8]) for i in range(n)]
                assert np.array_equal(d_dst[n - 1].cpu().numpy(), cv2.imdecode(np.frombuffer(want[m][(n - 1) % 8], np.uint8), 0))
                res["kb_per_frame_" + m] = round(sum(len(s) for s in want[m]) / 8 / 1e3, 1)
            enc_t = {m: [] for m in modes}
            deg_t = {m: [] for m in modes}
            for m, o in modes.items():           # warm-up
                dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), q, blob=(d_blob.data_ptr(), n * bound), optimize=o)
                dmc.degradeJPEG((d_src.data_ptr(), n, H, W), q, dst=d_dst.data_ptr(), optimize=o)
            torch.cuda.synchronize()
            for _ in range(5):
                for m, o in modes.items():
                    t0 = time.perf_counter()
                    dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), q, blob=(d_blob.data_ptr(), n * bound), optimize=o)
                    torch.cuda.synchronize(); enc_t[m].append(time.perf_counter() - t0)
                    t0 = time.perf_counter()
                    dmc.degradeJPEG((d_src.data_ptr(), n, H, W), q, dst=d_dst.data_ptr(), optimize=o)
                    torch.cuda.synchronize(); deg_t[m].append(time.perf_counter() - t0)
            for m in modes:
                res["encode_fps_" + m] = round(n / min(enc_t[m])); res["encode_fps_median_" + m] = round(n / float(np.median(enc_t[m])))
                res["degrade_roundtrip_fps_" + m] = round(n / min(deg_t[m])); res["degrade_roundtrip_fps_median_" + m] = round(n / float(np.median(deg_t[m])))
            # the decoder on per-frame-table streams from a host blob (the host parse is part of each call)
            hblob, hoffs = dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), q, optimize=True)
            hdst = np.empty((n, H, W), np.uint8)
            best, med = timed(lambda: dmc.jpegDecodeGrayBatch((hblob, hoffs), H, W, dst=hdst), 5)
            res["decode_host_blob_fps_optimize"] = round(n / best); res["decode_host_blob_fps_median_optimize"] = round(n / med)
            # cv2.imencode on all host threads (OpenCV releases the GIL)
            mm = 4 * threads
            for m, o in modes.items():
                enc = lambda i, o=o: cv2_enc(imgs[i % 8], q, o)
                list(pool.map(enc, range(threads)))
                t0 = time.perf_counter(); list(pool.map(enc, range(mm))); res["cv2_imencode_fps_all_threads_" + m] = round(mm / (time.perf_counter() - t0))
            out["sets"]["%s_q%d" % (kind, q)] = res
            print(kind, q, json.dumps(res), file=sys.stderr, flush=True)
            del d_blob
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
