"""pointcloudTest's frame loop (main.cpp:254-355) on batches, against the same loop through the single-frame public calls.
Writes one JSON record.

Loop per frame: prepare (depth16U2disp8U -> fillOcclusion -> transpose -> fillOcclusion -> transpose), code (degradeJPEG,
q80), filter (filterDisp8U2Depth32F(75, 575, 2.6, 1, 0, 1, 3, 65)), render (reprojectXYZ -> projectImagefromXYZ ->
fillSmallHole in place, isSub, three cameras: R = I with t = (+-100, 0, 0) and the "rot" view of tests/test_pointcloud.py,
K of main.cpp:132-136, exact division).  Sources at 1080p: 16-bit depth made from synth_disp frames (depth = FB * amp /
disparity, with holes of depth 0), and the tiled 16-bit Kinect crop.  The texture is a fixed colour image per frame.

  * batch path: device-resident frames through prepareDisparityBatch -> degradeJPEG -> chain_batch(DEPTH32F) ->
    renderViewBatch; frames/s and ms per frame of each stage (host clock, the device synchronised after each stage);
  * single-frame path: the same loop through the single-frame public calls from host memory, on a subset of the frames,
    alternating with the batch path in the same process; its views are compared with the batch path's;
  * preparation alone: prepareDisparityBatch (device and host memory) against the five single-image calls.

    python tools/pointcloud_batch.py [--frames 32] [--single 4] [--reps 3] [--out profiles/r10_pointcloud_batch.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import depthmapcompression_b200 as dmc                      # noqa: E402
from depthmapcompression_b200 import capi                   # noqa: E402
from oracle.oracle_py import synth_disp                     # noqa: E402
from _util import load_png                                  # noqa: E402
from test_pointcloud import VIEWS                           # noqa: E402

FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6
FB = FOCUS * BASELINE
CHAIN = (1, 0, 1, 3, 65.0)
QUALITY, F, H, W = 80, 1100.0, 1080, 1920


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    name, power, clock, cur = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "sm_clock_at_start": cur}


def cameras():
    rv = dict((n, (R, t)) for n, R, t in VIEWS)["rot"]
    return [(np.eye(3), np.array([100., 0., 0.])), (np.eye(3), np.array([-100., 0., 0.])), rv]


def intrinsics(f):
    K = np.eye(3) * f; K[0, 2] = (W - 1) * 0.5; K[1, 2] = (H - 1) * 0.5; K[2, 2] = 1.0
    return K


def sources(n):
    rs = np.random.RandomState(1)
    synth = []
    for i in range(n):
        d = synth_disp(H, W, 100 + i).astype(np.float64)
        z = np.rint(FB * AMP / d).astype(np.uint16)
        z[rs.rand(H, W) < 0.02] = 0
        z[200 + 3 * i:260 + 3 * i, 400:1500] = 0                   # a wide hole: rows that the fill blanks
        synth.append(z)
    crop = load_png("kinect_meeting_depth16_crop.png")
    tiled = np.tile(crop, (H // crop.shape[0] + 1, W // crop.shape[1] + 1))[:H, :W]
    kinect = [np.ascontiguousarray(np.roll(tiled, 37 * i, axis=1)) for i in range(n)]
    tex = np.stack([np.stack([(synth_disp(H, W, 500 + i) * k) & 255 for k in (1, 3, 7)], -1).astype(np.uint8) for i in range(n)])
    return {"synth_disp_1080p": np.stack(synth), "kinect_crop_tiled_1080p": np.stack(kinect)}, tex


def sync():
    dmc.default_context().synchronize()
    torch.cuda.synchronize()


class BatchPath:
    def __init__(self, d16, tex):
        self.n = len(d16)
        self.src = torch.from_numpy(d16.view(np.int16)).cuda()
        self.tex = torch.from_numpy(tex).cuda()
        self.disp = torch.empty((self.n, H, W), dtype=torch.uint8, device="cuda")
        self.dec = torch.empty_like(self.disp)
        self.depth = torch.empty((self.n, H, W), dtype=torch.float32, device="cuda")
        self.views = torch.empty((3, self.n, H, W, 3), dtype=torch.uint8, device="cuda")
        self.p = dmc.filters.chain_params(capi.CHAIN_DEPTH32F, *CHAIN, focus=FOCUS, baseline=BASELINE, amp=AMP)
        cams = cameras()
        self.R = np.stack([c[0] for c in cams]); self.t = np.stack([c[1] for c in cams]); self.K = intrinsics(F)

    def run(self):
        """-> seconds per stage"""
        n, ctx, out = self.n, dmc.default_context(), {}
        sync()
        t0 = time.perf_counter()
        dmc.prepareDisparityBatch((self.src.data_ptr(), n, H, W), FB, AMP, passes=2, dst=self.disp.data_ptr())
        sync(); t1 = time.perf_counter(); out["prepare"] = t1 - t0
        dmc.degradeJPEG((self.disp.data_ptr(), n, H, W), QUALITY, dst=self.dec.data_ptr())
        sync(); t2 = time.perf_counter(); out["code"] = t2 - t1
        ctx.chain_batch(self.dec.data_ptr(), self.depth.data_ptr(), n, H, W, self.p, device=True)
        sync(); t3 = time.perf_counter(); out["filter"] = t3 - t2
        dmc.renderViewBatch((self.depth.data_ptr(), n, H, W, np.float32), (self.tex.data_ptr(), n, H, W), F, self.R, self.t, self.K,
                            isSub=True, exact_divide=True, dst=self.views.data_ptr())
        sync(); out["render"] = time.perf_counter() - t3
        return out


def prepare_single(d16):
    x = dmc.depth16U2disp8U(d16, None, FB, AMP, 0.0)
    dmc.fillOcclusion(x, 0, dmc.FILL_DISPARITY)
    return dmc.transpose(dmc.fillOcclusion(dmc.transpose(x), 0, dmc.FILL_DISPARITY))


def single_path(d16, tex):
    """The loop through the single-frame public calls from host memory -> (seconds per stage, views [3, n, H, W, 3])"""
    pfs = dmc.PostFilterSet()
    cams, K = cameras(), intrinsics(F)
    views = np.empty((3, len(d16), H, W, 3), np.uint8)
    tm = dict.fromkeys(("prepare", "code", "filter", "render"), 0.0)
    for i in range(len(d16)):
        t0 = time.perf_counter()
        disp = prepare_single(d16[i])
        t1 = time.perf_counter()
        dec, _ = dmc.degradeJPEG(disp, QUALITY)
        t2 = time.perf_counter()
        depth = pfs.filterDisp8U2Depth32F(dec, None, FOCUS, BASELINE, AMP, *CHAIN)
        t3 = time.perf_counter()
        for v, (R, t) in enumerate(cams):
            xyz = dmc.reprojectXYZ(depth, None, F)
            views[v, i] = dmc.fillSmallHole(dmc.projectImagefromXYZ(tex[i], None, xyz, R, t, K, isSub=True, exact_divide=True))
        t4 = time.perf_counter()
        for k, a, b in (("prepare", t0, t1), ("code", t1, t2), ("filter", t2, t3), ("render", t3, t4)):
            tm[k] += b - a
    return tm, views


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--single", type=int, default=4, help="frames of the single-frame path (a subset of the batch)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_pointcloud_batch.json"))
    a = ap.parse_args()
    rec = {"gpu": gpu_info(), "frames": a.frames, "single_frames": a.single, "reps": a.reps, "quality": QUALITY, "chain": list(CHAIN),
           "cameras": 3, "isSub": True, "exact_divide": True, "f": F, "size": [H, W], "sources": {}}
    srcs, tex = sources(a.frames)
    for name, d16 in srcs.items():
        bp = BatchPath(d16, tex)
        bp.run()                                        # warm-up: modules, scratch, tables
        single_path(d16[:1], tex[:1])
        batch_t, single_t = [], []
        for _ in range(a.reps):                         # alternating in one process
            batch_t.append(bp.run())
            tm, views = single_path(d16[:a.single], tex[:a.single])
            single_t.append(tm)
        same = bool(np.array_equal(bp.views[:, :a.single].cpu().numpy(), views))
        best_b = min(batch_t, key=lambda r: sum(r.values()))
        best_s = min(single_t, key=lambda r: sum(r.values()))
        r = {"batch": {"frames_per_s": a.frames / sum(best_b.values()), "ms_per_frame": {k: 1e3 * v / a.frames for k, v in best_b.items()},
                       "ms_per_rendered_view": 1e3 * best_b["render"] / (3 * a.frames)},
             "single": {"frames_per_s": a.single / sum(best_s.values()), "ms_per_frame": {k: 1e3 * v / a.single for k, v in best_s.items()}},
             "views_equal_single_vs_batch": same}
        r["speedup"] = r["batch"]["frames_per_s"] / r["single"]["frames_per_s"]
        # preparation alone: batched (device, host) against the five single-image calls
        host_out = np.empty((a.frames, H, W), np.uint8)
        dmc.prepareDisparityBatch(d16, FB, AMP, passes=2, dst=host_out)
        pd, ph, ps = [], [], []
        for _ in range(a.reps):
            sync(); t0 = time.perf_counter()
            dmc.prepareDisparityBatch((bp.src.data_ptr(), a.frames, H, W), FB, AMP, passes=2, dst=bp.disp.data_ptr())
            sync(); pd.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            dmc.prepareDisparityBatch(d16, FB, AMP, passes=2, dst=host_out)
            ph.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            single = [prepare_single(d16[i]) for i in range(a.single)]
            ps.append((time.perf_counter() - t0) / a.single * a.frames)
        r["prepare"] = {"batch_device_ms_per_frame": 1e3 * min(pd) / a.frames, "batch_host_ms_per_frame": 1e3 * min(ph) / a.frames,
                        "single_calls_ms_per_frame": 1e3 * min(ps) / a.frames,
                        "equal": bool(all(np.array_equal(single[i], host_out[i]) for i in range(a.single)))}
        rec["sources"][name] = r
        print(name, json.dumps(r, indent=1), flush=True)
        del bp
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
