#!/usr/bin/env python
"""bench.py -- headline benchmark of the post filter set on B200 (contract in the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

--dump-outputs DIR writes, after the timed steps, the filtered frames the last timed step produced for a fixed seeded
sample of each rank's frames, as float32 DIR/filtered_frames.npy ([frames, 1080, 1920]; DIR/filtered_frames_rank<r>.npy
with several ranks), at most 64 MB (64e6 bytes) in all.  The inputs depend only on the arguments, so two builds can be compared
output for output.

Workload (BASELINE.json configs[2]): a 1920x1080 8-bit x264-decoded disparity video of 1000 frames per GPU, full chain
PostFilterSet::operator()(median_r=2, gaussian_r=1, minmax_r=3, brange_r=5, brange_th=10).  The frames are built from the
reference's own x264-decoded frame (tests/golden/x264_depth_y.png = the Y plane of its bundled depth.yuv) tiled 3x3 to
1080p and translated by (f, 2f) pixels in frame f, so that every frame carries real codec texture (SURVEY.md 8d).  A "step" is one pass
of the chain over the rank's 1000 frames (2.07 GB in, 2.07 GB out: far larger than the 126 MB L2, so no L2
flush is needed between steps).  Frames are sharded frame-parallel: every rank owns its own frames, no collective
on the data path ("scaling": "weak").

  value   Mpixel/s of the whole job with frames resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e     the same metric through the public streaming entry point dmc_chain_batch with pinned HOST buffers:
          H2D copy of every input frame and D2H copy of every output frame inside the timed region
  roofline  the dominant kernel (8-bit binary-weighted range filter): algorithmic bytes (2 B/pixel) / its mean
          launch duration measured live with CUDA events around each launch, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the reference's own CPU code (oracle/_ref, unmodified sources through the cv:: shim) on the host cores,
          frame-parallel over all hardware threads, on a bounded sample of the same frames
  e2e_bitstream  the same chain fed with JPEG bitstreams of the frames (dmc_chain_batch_jpeg: decode on the GPU, bit-exact
          with cv::imdecode; about 1/30 of the host-to-device bytes), host pinned -> host pinned
  strong_scaling  configs[2] read literally: 1000 frames in total, sharded over the ranks (device-resident)
  sched_e2e  the in-process frame-batch scheduler (dmc_sched_*) driven by rank 0 over every GPU of the job, host -> host

--impl reference times that CPU path as the run's subject (same metric / config), rank 0 only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 1080, 1920
CHAIN = dict(median_r=2, gaussian_r=1, minmax_r=3, brange_r=5, brange_th=10)
ALGO_BYTES_PER_PX = 2.0            # operator(): 1 B read + 1 B written per pixel (SURVEY.md 8d)
HBM_FALLBACK_GBS = 6650.0          # /opt/skills/guides/B200_PROFILING.md fallback
DATA_NOTE = "synthetic video: the reference's x264-decoded depth frame (depth.yuv Y plane, golden fixture) tiled to 1080p and translated per frame"


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ the video
def base_frame():
    """The reference's x264-decoded disparity frame (Y plane of depth.yuv, x264FFMPEGDemo.cpp:22-35; committed as a golden
    fixture) tiled 3x3 and cropped to 1920x1080."""
    import cv2
    y = cv2.imread(os.path.join(ROOT, "tests", "golden", "x264_depth_y.png"), cv2.IMREAD_UNCHANGED)
    assert y is not None and y.shape == (480, 640) and y.dtype == np.uint8
    return np.ascontiguousarray(np.tile(y, (3, 3))[:H, :W])


def frame_np(base, f):
    """frame f of the video: the base frame translated by (f, 2f) pixels with wrap-around"""
    return np.roll(base, (f % H, (2 * f) % W), axis=(0, 1))


def make_frames_torch(n, first, device):
    """frames first .. first+n-1 of the video, built on the device"""
    import torch
    b = torch.from_numpy(base_frame()).to(device)
    out = torch.empty((n, H, W), dtype=torch.uint8, device=device)
    for i in range(n):
        f = first + i
        out[i] = torch.roll(b, shifts=(f % H, (2 * f) % W), dims=(0, 1))
    return out


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []; self.proc = None; self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for nme, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def cpu_chain_throughput(frames, budget_s=12.0, prefer_reference=True):
    """Times the reference's CPU implementation of the chain on `frames` (numpy [n, H, W] uint8), frame-parallel over
    all host threads (each worker runs the chain single-threaded: frames are independent, which is how a user of the
    reference would use every core on a video).  Returns (Mpixel/s, info dict)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle_py
    lib, kind = None, "port"
    if prefer_reference and oracle_py.Reference.available():
        try:
            lib = oracle_py.Reference(); kind = "reference"
        except Exception:
            lib = None
    if lib is None:
        lib = oracle_py.Port(); kind = "port"
    cores = os.cpu_count() or 1
    p = CHAIN

    def work(i):
        lib.set_num_threads(1)          # OpenMP ICV is per calling thread
        return lib.post_filter_set(frames[i % len(frames)], p["median_r"], p["gaussian_r"], p["minmax_r"], p["brange_r"], p["brange_th"])

    with ThreadPoolExecutor(cores) as ex:
        t0 = time.perf_counter(); list(ex.map(work, range(cores))); t1 = time.perf_counter()      # warm-up + calibration
        per_round = max(t1 - t0, 1e-3)
        rounds = int(max(1, min(2000, budget_s / per_round)))
        n = rounds * cores
        t0 = time.perf_counter(); list(ex.map(work, range(n))); t1 = time.perf_counter()
    wall = t1 - t0
    mpix = n * H * W / wall / 1e6
    # the reference's own intra-frame parallelism (cv::parallel_for_ in the range filter only), for the record
    lib.set_num_threads(0)
    t0 = time.perf_counter()
    for i in range(2):
        lib.post_filter_set(frames[i % len(frames)], p["median_r"], p["gaussian_r"], p["minmax_r"], p["brange_r"], p["brange_th"])
    intra = 2 * H * W / (time.perf_counter() - t0) / 1e6
    info = {"value": round(mpix, 2), "unit": "Mpixel/s", "cores": cores, "kind": kind, "sample_wall_s": round(wall, 2), "sample_frames": n,
            "sample": "%d frames of 1920x1080 (frames of the benchmark's own video), frame-parallel on %d threads, %.1f s" % (n, cores, wall),
            "intra_frame_parallel_mpix_s": round(intra, 2), "cpu_model": cpu_model()}
    if kind == "reference":
        info["third_party_stages"] = third_party_stage_times(lib, frames[0], p)
    return mpix, info


def third_party_stage_times(lib, frame, p, reps=3):
    """SURVEY 8(d): the reference calls OpenCV for the median, the Gaussian and dilate/erode; oracle/_ref compiles it against
    SSE stand-ins.  Times those stages one-threaded in both forms, so that the reader can see how much of the CPU chain the
    stand-ins account for and what the chain would cost with real OpenCV (cv2) underneath."""
    def t(f):
        f(); t0 = time.perf_counter()
        for _ in range(reps): f()
        return (time.perf_counter() - t0) / reps * 1e3
    lib.set_num_threads(1)
    km, kg, ks = 2 * p["median_r"] + 1, 2 * p["gaussian_r"] + 1, 2 * p["minmax_r"] + 1
    out = {"chain_ms_per_frame_1thr": round(t(lambda: lib.post_filter_set(frame, p["median_r"], p["gaussian_r"], p["minmax_r"], p["brange_r"], p["brange_th"])), 1),
           "standins_ms": round(t(lambda: lib.median_blur(frame, km)) + t(lambda: lib.small_gaussian(frame, kg, p["gaussian_r"] + 0.5)) +
                                t(lambda: lib.morph(frame, ks, 1)) + t(lambda: lib.morph(frame, ks, 0)), 1)}
    try:
        import cv2
        cv2.setNumThreads(1)
        k = np.ones((ks, ks), np.uint8)
        def gauss():
            f = frame.astype(np.float32); g = cv2.GaussianBlur(f, (kg, kg), p["gaussian_r"] + 0.5); return np.rint(g).astype(np.uint8)
        out["cv2_ms"] = round(t(lambda: cv2.medianBlur(frame, km)) + t(gauss) + t(lambda: cv2.dilate(frame, k)) + t(lambda: cv2.erode(frame, k)), 1)
        out["chain_ms_with_cv2_stages"] = round(out["chain_ms_per_frame_1thr"] - out["standins_ms"] + out["cv2_ms"], 1)
        out["cv2_version"] = cv2.__version__
    except Exception as e:      # cv2 missing: the stand-in figures stand alone
        out["cv2"] = "unavailable (%s)" % type(e).__name__
    return out


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def config_dict(n_gpus, frames_per_gpu):
    return {"devices": None, "workload": "configs[2]: 1920x1080 8UC1 x264-decoded disparity video (the reference's depth.yuv frame tiled 3x3, translated per frame), %d frames per GPU, PostFilterSet::operator()(2,1,3,5,10) FULL_KERNEL" % frames_per_gpu,
            "frames_per_gpu": frames_per_gpu, "height": H, "width": W, "chain": CHAIN,
            "l2": "inputs (%.2f GB per step per GPU) larger than the 126 MB L2; no flush" % (frames_per_gpu * H * W / 1e9),
            "parallelism": "frame-parallel x%d, no collective" % n_gpus}


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, d_out, rank, world):
    """Writes the frames of d_out (the device-resident output of the last timed step) at a seeded sample of frame
    indices, as float32; the ranks share the DUMP_BYTES budget (with more ranks than frames fit, the last ranks write none)."""
    n = d_out.shape[0]
    total = min(world * n, DUMP_BYTES // (H * W * 4))
    k = total // world + (1 if rank < total % world else 0)
    if k == 0:
        return
    idx = np.sort(np.random.RandomState(0).choice(n, k, replace=False))
    frames = d_out[idx.tolist()].cpu().numpy().astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "filtered_frames.npy" if world == 1 else "filtered_frames_rank%d.npy" % rank), frames)


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=1000, help="frames per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lanes", type=int, default=1, help="frame groups in flight on separate streams (device-resident path)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's output frames to DIR (float32 .npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3:
        args.warmup = 3

    if args.impl == "reference":
        if rank != 0:
            return
        base = base_frame()
        frames = np.stack([frame_np(base, f) for f in (0, 1, 333, 500, 998, 999, 7, 13)])      # the frames our arm's parity gate samples
        vals, walls, nfr = [], [], []
        for it in range(args.warmup + args.steps):
            mp, info = cpu_chain_throughput(frames, budget_s=max(2.0, 60.0 / (args.warmup + args.steps)))
            if it >= args.warmup:
                vals.append(mp); walls.append(info["sample_wall_s"]); nfr.append(info["sample_frames"])
        v = float(np.mean(vals)); info["value"] = round(v, 2)
        # every step is a bounded SAMPLE of the 1000-frame workload (the CPU needs about 4 s per 1000 frames per 16 threads x 60);
        # ms_per_step is derived from the measured rate, the measured wall time of each sample is listed next to it
        info["sampled"] = True; info["sample_wall_s_per_step"] = walls; info["sample_frames_per_step"] = nfr
        line = {"impl": "reference", "metric": "Mpixel/s of full post-filter chain (1080p)", "value": round(v, 2), "unit": "Mpixel/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(args.frames * H * W / (v * 1e6) * 1e3, 3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": DATA_NOTE,
                "config": config_dict(args.gpus, args.frames), "cpu_baseline": info, "sampled": True,
                "ms_per_step_note": "derived: frames of one step / measured rate; each step timed a sample of %s frames in %s s" % (nfr, [round(w, 1) for w in walls]),
                "e2e": {"value": round(v, 2), "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line)); return

    import torch
    import torch.distributed as dist
    import depthmapcompression_b200 as dmc
    from depthmapcompression_b200 import capi
    from depthmapcompression_b200.filters import chain_params
    # Which GPU does rank r use?  On a box with more GPUs than ranks the host links are not equal (profiles/r02_hostlink.json:
    # GPUs 0-3 of this pool's boxes share an upstream that carries ~51 GB/s each way, GPUs 4-7 one that carries ~94), so rank 0
    # measures every visible device's link once (all devices copying both ways at the same time, ~0.3 s) and the job takes the
    # `world` devices with the fastest links.  DMC_BENCH_DEVICES=0,1,.. pins the choice; with as many ranks as GPUs it is moot.
    vis = torch.cuda.device_count()
    if world > 1:
        dist.init_process_group("cpu:gloo,cuda:nccl")              # objects travel over gloo, CUDA tensors over NCCL
    devmap = list(range(world)); devmap_how = "rank r on device r"
    if os.environ.get("DMC_BENCH_DEVICES"):
        devmap = [int(x) for x in os.environ["DMC_BENCH_DEVICES"].split(",")][:world]; devmap_how = "DMC_BENCH_DEVICES"
    elif vis > world:
        if rank == 0:
            try:
                pr = dmc.hostlink_probe(list(range(vis)))
                order = sorted(range(vis), key=lambda d: (-pr["loaded_gbs"][d], d))
                devmap = sorted(order[:world]); devmap_how = "the %d of %d visible devices with the fastest host links (GB/s each way, all devices loaded: %s)" % (world, vis, pr["loaded_gbs"])
            except Exception as ex:
                devmap_how = "rank r on device r (link probe failed: %s)" % ex
            for d in range(vis):                                   # the probe left a CUDA context on every device: give back the ones rank 0 does not use
                if d != devmap[0]:
                    capi.lib.dmc_release_device(d)
        if world > 1:
            box = [(devmap, devmap_how)]; dist.broadcast_object_list(box, src=0, device=torch.device("cpu")); devmap, devmap_how = box[0]
    local = devmap[rank % len(devmap)]
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ctx = dmc.Context(local)
    stream = torch.cuda.Stream(device=dev)             # a real (non-default) stream: the kernels and the timing events share it
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_lanes(args.lanes)
    N = args.frames
    p = chain_params(capi.CHAIN_DISP8U, **CHAIN)
    d_in = make_frames_torch(N, rank * N, dev)                  # rank r owns frames r*N .. r*N+N-1 of the video
    d_out = torch.zeros_like(d_in)
    torch.cuda.synchronize()

    # parity gate: 8 frames of this very input against the CPU oracle (rank 0 keeps the frames for the CPU baseline)
    sample_idx = [0, 1, N // 3, N // 2, N - 2, N - 1, 7 % N, 13 % N]
    ctx.chain_batch(d_in.data_ptr(), d_out.data_ptr(), N, H, W, p, device=True); ctx.synchronize()
    sample_in = d_in[sample_idx].cpu().numpy()
    # every rank checks its own frames (different seeds, different devices) and the verdicts are all-reduced: a wrong
    # result on any GPU aborts the whole run before anything is timed
    from oracle.oracle_py import Port
    port = Port(); port.set_num_threads(max(1, (os.cpu_count() or 1) // world)); got = d_out[sample_idx].cpu().numpy()
    bad = 0
    for i in range(len(sample_idx)):
        want = port.post_filter_set(sample_in[i], CHAIN["median_r"], CHAIN["gaussian_r"], CHAIN["minmax_r"], CHAIN["brange_r"], CHAIN["brange_th"])
        if not np.array_equal(got[i], want):
            bad += 1; print("rank %d: parity gate failed on frame %d" % (rank, sample_idx[i]), file=sys.stderr)
    if world > 1:
        tb = torch.tensor([bad], device=dev, dtype=torch.int32); dist.all_reduce(tb, op=dist.ReduceOp.SUM); bad = int(tb[0])
    if bad:
        raise SystemExit("parity gate failed on %d sampled frames (all ranks)" % bad)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def run_step():
        ctx.chain_batch(d_in.data_ptr(), d_out.data_ptr(), N, H, W, p, device=True)

    for _ in range(args.warmup):
        run_step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ctx.profile_read(capi.STAGE_RANGE, reset=True)
    ctx.profile_enable(1 << capi.STAGE_RANGE)          # two event records per range-filter launch
    l0 = ctx.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        run_step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.kernel_launches - l0
    rng_ms, rng_n, rng_px = ctx.profile_read(capi.STAGE_RANGE, reset=True)
    ctx.profile_enable(0)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms, float(launches)], device=dev, dtype=torch.float64)
    if world > 1:
        tm = t.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = t.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        ms = float(tm[0]); launches = int(ts[1])
    ms_per_step = ms / args.steps
    value = world * N * H * W / (ms_per_step * 1e-3) / 1e6
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d_out, rank, world)

    # stage breakdown (untimed extra pass with every stage bracketed)
    ctx.profile_enable(15)
    for s in range(4):
        ctx.profile_read(s, reset=True)
    run_step(); ctx.synchronize()
    stage_ms = {capi.STAGE_NAMES[s]: round(ctx.profile_read(s, reset=True)[0], 3) for s in range(4)}
    ctx.profile_enable(0)

    # end to end through the public streaming entry point with pinned host buffers
    ctx.set_stream(None)
    h_in = torch.empty((N, H, W), dtype=torch.uint8).pin_memory()
    h_out = torch.empty((N, H, W), dtype=torch.uint8).pin_memory()
    h_in.copy_(d_in.cpu())

    def e2e_run(steps):
        for _ in range(2):
            ctx.chain_batch(h_in.data_ptr(), h_out.data_ptr(), N, H, W, p, device=False)
        barrier()
        t0 = time.perf_counter(); step_ms = []
        for _ in range(steps):
            ts = time.perf_counter()
            ctx.chain_batch(h_in.data_ptr(), h_out.data_ptr(), N, H, W, p, device=False)     # returns when h_out is valid
            step_ms.append(round((time.perf_counter() - ts) * 1e3, 2))
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([secs], device=dev, dtype=torch.float64); dist.all_reduce(tt, op=dist.ReduceOp.MAX); secs = float(tt[0])
        if not torch.equal(h_out[sample_idx], d_out[sample_idx].cpu()):
            raise SystemExit("e2e output differs from the device-resident output")
        return world * N * H * W * steps / secs / 1e6, step_ms

    e2e_steps = max(2, min(args.steps, 5))
    # (1) every rank on its own device's link
    e2e_own, own_step_ms = e2e_run(e2e_steps)
    # (2) topology-aware: rank 0 measures the host link of the job's devices while every rank is idle (all devices copying
    # both ways at once, then the best subset alone) and proposes which links should carry the traffic; ranks whose link is
    # not worth using stage through a gateway device's HBM and reach it over NVLink (dmc_set_gateway).  Same bytes, same
    # results; on a box with uniform links nothing is re-routed and (2) == (1).
    barrier()
    link = None
    if rank == 0:
        try:
            link = dmc.hostlink_probe(devmap)
        except Exception as ex:      # a probe failure must not take the benchmark down: everybody keeps its own link
            link = {"error": str(ex), "gateway": list(devmap), "all_gbs": None, "best_gbs": None, "loaded_gbs": [], "n_link": world}
    torch.cuda.set_device(local)
    if world > 1:
        box = [link]; dist.broadcast_object_list(box, src=0, device=torch.device("cpu")); link = box[0]
    routed = link["gateway"][rank] != local if world > 1 else False
    any_routed = any(link["gateway"][r] != devmap[r] for r in range(world))
    e2e_value, e2e_step_ms = e2e_own, own_step_ms
    if any_routed:
        if routed:
            ctx.set_gateway(link["gateway"][rank])
        e2e_value, e2e_step_ms = e2e_run(e2e_steps)
        if routed:
            ctx.set_gateway(-1)
    if e2e_own > e2e_value:          # the routing has to earn its keep
        e2e_value, e2e_step_ms, any_routed = e2e_own, own_step_ms, False
    h_out_ref = h_out[:8].clone()      # filtered frames 0..7 of this rank (the scheduler check below compares against them)

    # ---- e2e from JPEG bitstreams: the reference's own ingest (cv::imdecode, main.cpp:284) moved onto the GPU -- the host link
    # carries the coded frames (a few % of the raw bytes) in and the filtered frames out
    e2e_bits = None
    try:
        import cv2
        NU = 64                                                    # distinct coded frames; the 1000-frame batch cycles through them
        raw = d_in[:NU].cpu().numpy()
        coded = [cv2.imencode(".jpg", raw[i], [cv2.IMWRITE_JPEG_QUALITY, 80])[1].tobytes() for i in range(NU)]
        decoded = np.stack([cv2.imdecode(np.frombuffer(c, np.uint8), 0) for c in coded[:4]])
        want4 = np.stack([port.post_filter_set(decoded[i], CHAIN["median_r"], CHAIN["gaussian_r"], CHAIN["minmax_r"], CHAIN["brange_r"], CHAIN["brange_th"]) for i in range(4)])
        blob, offsets = dmc.pack_streams([coded[i % NU] for i in range(N)])
        h_blob = torch.empty(blob.size, dtype=torch.uint8).pin_memory(); h_blob.numpy()[:] = blob
        if any_routed and routed:                                  # the routing that won the raw run carries this one too
            ctx.set_gateway(link["gateway"][rank])
        for _ in range(2):
            ctx.chain_batch_jpeg((h_blob.data_ptr(), offsets), H, W, h_out.data_ptr(), p)
        if not np.array_equal(h_out[:4].numpy(), want4):
            raise SystemExit("bitstream e2e differs from cv2.imdecode + oracle chain")
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            ctx.chain_batch_jpeg((h_blob.data_ptr(), offsets), H, W, h_out.data_ptr(), p)
        torch.cuda.synchronize(); secs = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([secs], device=dev, dtype=torch.float64); dist.all_reduce(tt, op=dist.ReduceOp.MAX); secs = float(tt[0])
        if any_routed and routed:
            ctx.set_gateway(-1)
        e2e_bits = {"value": round(world * N * H * W * e2e_steps / secs / 1e6, 1), "unit": "Mpixel/s", "steps": e2e_steps, "routing": (link["gateway"] if any_routed else "own links"),
                    "h2d_bytes_per_step": int(world * blob.size), "d2h_bytes_per_step": world * N * H * W,
                    "api": "dmc_chain_batch_jpeg(host pinned JPEG q80 bitstreams -> decode on the GPU -> chain -> host pinned)",
                    "kb_per_frame": round(blob.size / N / 1e3, 1), "parity": "first 4 frames == oracle chain on cv2.imdecode of the same streams"}
    except SystemExit:
        raise
    except Exception as ex:                                        # cv2 missing on the box: the key says so instead of the run dying
        e2e_bits = {"unavailable": "%s: %s" % (type(ex).__name__, ex)}
        if world > 1:
            tt = torch.tensor([0.0], device=dev, dtype=torch.float64); dist.all_reduce(tt, op=dist.ReduceOp.MAX)

    # ---- strong scaling: configs[2] read literally -- 1000 frames in TOTAL, sharded over the ranks (device-resident)
    lo, cnt = capi.shard_frames(N, rank, world)
    def run_shard():
        if cnt:
            ctx.chain_batch(d_in.data_ptr(), d_out.data_ptr(), cnt, H, W, p, device=True)
    ctx.set_stream(stream.cuda_stream)
    for _ in range(2):
        run_shard()
    barrier(); e0.record(stream)
    for _ in range(args.steps):
        run_shard()
    e1.record(stream); barrier()
    sms = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([sms], device=dev, dtype=torch.float64); dist.all_reduce(tt, op=dist.ReduceOp.MAX); sms = float(tt[0])
    strong = {"frames_total": N, "frames_per_rank": [capi.shard_frames(N, r, world)[1] for r in range(world)], "ms_per_step": round(sms / args.steps, 3),
              "value": round(N * H * W * args.steps / (sms * 1e-3) / 1e6, 1), "unit": "Mpixel/s", "scaling": "strong"}
    ctx.set_stream(None)

    # ---- the in-process frame-batch scheduler (dmc_sched_*), rank 0 drives every GPU of the job, the other ranks idle
    sched = None
    barrier()
    if rank == 0:
        try:
            NS = min(N, 400)                                       # frames per device (pinned host memory: 2 x 0.83 GB per device)
            devs = list(devmap)
            fbs = dmc.FrameBatchScheduler(devs)
            s_in = torch.empty((NS * world, H, W), dtype=torch.uint8).pin_memory(); s_out = torch.empty_like(s_in).pin_memory()
            for dv in range(world):
                s_in[dv * NS:(dv + 1) * NS].copy_(h_in[:NS])
            for _ in range(2):
                fbs.chain_batch(s_in.data_ptr(), s_out.data_ptr(), NS * world, H, W, p)
            ok = all(torch.equal(s_out[dv * NS:dv * NS + 8], h_out_ref[:8]) for dv in range(world))
            ts = []
            for _ in range(3):
                t0 = time.perf_counter(); fbs.chain_batch(s_in.data_ptr(), s_out.data_ptr(), NS * world, H, W, p); ts.append(time.perf_counter() - t0)
            gw, own_gbs, routed_gbs = fbs.routing()
            sched = {"value": round(NS * world * H * W / min(ts) / 1e6, 1), "unit": "Mpixel/s", "devices": devs, "frames": NS * world, "ms": [round(t * 1e3, 2) for t in ts],
                     "bit_exact_vs_chain_batch": bool(ok), "routing": gw, "link_gbs_own": own_gbs, "link_gbs_routed": routed_gbs,
                     "api": "dmc_sched_chain_batch (one process, one host thread + context per device, host pinned -> host pinned)"}
            del fbs, s_in, s_out
        except Exception as ex:
            sched = {"unavailable": "%s: %s" % (type(ex).__name__, ex)}
        torch.cuda.set_device(local)
    barrier()

    if rank == 0:
        peak, peak_src = hbm_peak()
        roof = None
        if rng_n:
            dur_s = rng_ms * 1e-3 / rng_n
            bytes_per_launch = ALGO_BYTES_PER_PX * rng_px / rng_n
            ach = bytes_per_launch / dur_s / 1e9
            traffic = None; issue = None
            try:
                with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                    tj = json.load(f)      # ncu DRAM bytes of one captured launch, scaled to this run's mean launch size
                    traffic = int(tj["range_filter_dram_bytes_per_launch"] * bytes_per_launch / tj["algorithmic_bytes_per_launch"])
                    if "issue_active_pct" in tj:       # what actually bounds the kernel (from the same ncu capture, not live)
                        issue = {k: tj[k] for k in ("lane_instructions_per_pixel", "issue_active_pct", "pipe_alu_pct", "pipe_fma_pct")}
                        issue["source"] = "profiles/traffic.json (ncu --set full)"
            except Exception:
                pass
            roof = {"bound": "hbm", "kernel": "range filter (bwrf8u)", "achieved": round(ach, 2), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 5),
                    "traffic": traffic, "peak_source": peak_src, "launches_timed": int(rng_n), "mean_launch_ms": round(dur_s * 1e3, 4),
                    "algorithmic_bytes_per_launch": int(bytes_per_launch), "issue": issue, "share_of_step": round(rng_ms / ms if world == 1 else rng_ms / (ms_per_step * args.steps), 4),
                    "note": "instruction-bound stencil (about 220 lane-instructions per pixel for 81 taps, 85 % of the issue slots): HBM fraction is small by construction, see DESIGN.md"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            _, cpu = cpu_chain_throughput(sample_in, budget_s=12.0)
        line = {"metric": "Mpixel/s of full post-filter chain (1080p)", "value": round(value, 1), "unit": "Mpixel/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": DATA_NOTE, "config": dict(config_dict(world, N), devices=devmap, devices_chosen_by=devmap_how, visible_devices=vis), "clocks": clocks,
                "e2e": {"value": round(e2e_value, 1), "unit": "Mpixel/s", "h2d_bytes_per_step": world * N * H * W, "d2h_bytes_per_step": world * N * H * W,
                        "steps": e2e_steps, "step_ms": e2e_step_ms, "api": "dmc_chain_batch(host pinned -> host pinned), 4-slot H2D/kernel/D2H pipeline",
                        "own_links_value": round(e2e_own, 1), "routing": (link["gateway"] if any_routed else "own links"),
                        "link_ceiling_gbs": link.get("best_gbs"), "link_all_devices_gbs": link.get("all_gbs"), "link_loaded_gbs_per_device": link.get("loaded_gbs"),
                        "frac_of_link": (round(e2e_value * 1e-3 / link["best_gbs"], 3) if link.get("best_gbs") else None),
                        "link_note": "ceiling = GB/s each way measured by dmc_hostlink_probe in this run (64 MB copies both ways on the job's devices at once; best of all devices / the proposed link set); the chain moves 1 B/pixel each way"},
                "e2e_bitstream": e2e_bits, "strong_scaling": strong, "sched_e2e": sched,
                "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "stage_ms_per_step": stage_ms,
                "fps_1080p": round(value * 1e6 / (H * W), 1)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
