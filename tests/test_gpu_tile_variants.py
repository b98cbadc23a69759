"""The launch-size variants of the tiled kernels on the chain's hot path, against the CPU oracle.

Every tiled kernel is compiled in several shapes, and its launcher picks one from the launch: fewer than 2 x 148 tiles
(the frame count included) take short tiles, larger launches the full ones; W and the dst address pick 2- or 4-byte
stores or byte stores; the threshold picks the 8-bit range filter's FLUSH accumulator, the source type and threshold
the 32-bit range filter's accumulation MODE.  Each variant is its own unrolled body with its own partial-tile guards,
so each can be wrong on its own.

`variant_*` below restate the launchers' rules; TABLE lists every instantiation some input can reach.  CASES reaches
every entry of TABLE, mostly through frame batches of small frames (many frames put a small frame size into the full
variants cheaply), and every output is compared bit for bit with the oracle.  test_profiler_names checks the rules
against the kernel names the profiler records.  Only the two table tests run without a GPU; run the rest with
`-m gpu` on a B200."""
import json
import re
from typing import NamedTuple

import numpy as np
import pytest

from _util import assert_bits_equal, make_image, mask_undefined, ntaps

SMS = 148
FEW_TILES = 2 * SMS                 # a launch with fewer tiles takes the short-tile variant
TILE_W = 128
CHAIN_DISP8U, CHAIN_DEPTH32F, CHAIN_DEPTH16U, CHAIN_DISP32F = 0, 1, 2, 3
FULL_KERNEL = 0
FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6
GROUP_MB = 256                      # default DMC_GROUP_MB of dmc_chain_batch


# ---------------------------------------------------------------------------------------------- the launchers' rules
def tiles(n, H, W, tile_h):
    return -(-W // TILE_W) * -(-H // tile_h) * n


def variant_median(r, n, H, W, dst):
    """launch_median8u_fast (dmc_front8u.cu): 3x3 / 5x5 circuits decide with 32-row tiles, bisection always R = 4"""
    if not 1 <= r <= 10:
        return None
    even = W % 2 == 0 and dst % 2 == 0
    if r >= 3:
        return ("median8u_bisect", r, 4, even)
    return ("median8u_p2", r, 2 if tiles(n, H, W, 32) < FEW_TILES else 16, even)


def variant_gauss(gr, n, H, W, dst):
    """launch_gauss8u_fast for the chain's d = 2 gr + 1: a 1-pixel-high or -wide image drops one pass (generic kernel)"""
    if gr not in (1, 2) or H == 1 or W == 1:
        return None
    R = 2 if tiles(n, H, W, 64) < FEW_TILES else (8 if gr == 1 else 4)
    return ("gauss8u_p4", gr, R, W % 4 == 0 and dst % 4 == 0)


def variant_minmax(r, n, H, W, dst):
    """launch_minmax_rad: decides with 64-row tiles"""
    if not 1 <= r <= 5:
        return None
    return ("minmax8u_p2", r, 4 if tiles(n, H, W, 64) < FEW_TILES else 16, W % 2 == 0 and dst % 2 == 0)


def th8(threshold):
    return int(threshold) & 0xFF     # (uchar)threshold (range_filter_8u)


def variant_bwrf8u(r, threshold, n, H, W, dst, cn=1):
    """launch_bwrf8u_h2 / launch_bwrf8u_c3_h2: the packed path needs (2r+1) * th <= 2048"""
    th = th8(threshold)
    if cn == 3:
        if not 1 <= r <= 7 or (2 * r + 1) * th > 2048:
            return None
        return ("bwrf8u_c3_h2", r, 4 if r <= 2 else (2 if r <= 5 else 1), ntaps(r) * th > 2048)
    if not 1 <= r <= 10 or (2 * r + 1) * th > 2048:
        return None
    R = 8 if r <= 3 else (4 if r <= 6 else (2 if r <= 8 else 1))
    if R > 2 and tiles(n, H, W, 4 * R) < FEW_TILES:
        R = 2
    return ("bwrf8u_h2", r, R, ntaps(r) * th > 2048, W % 2 == 0 and dst % 2 == 0)


def variant_bwrf32f(r, th, load, n, H, W, cn=1):
    """launch_bwrf32f_tiled / launch_bwrf32f_c3_tiled; load is "f32", "u16", "s16", "u8" or "u8disp" (the fused
    disparity -> depth load)"""
    if not 1 <= r <= 10:
        return None
    if cn == 3:
        if load not in ("f32", "u16", "s16"):
            return None
        R = 8 if r <= 3 else (4 if r <= 5 else (2 if r <= 7 else 1))
        fits = ((TILE_W + 2 * r) * 3 + 1) * (2 * R + 2 * r) * 4 <= 48 * 1024      # static shared memory
        return ("bwrf32f_c3_tiled", r, R if fits else R // 2)
    integer = load in ("u16", "s16", "u8") and th >= 0 and r <= 9
    mode = (2 if load == "s16" else 1) if integer else 0
    if mode == 0:
        R = 8 if r <= 3 else (4 if r <= 5 else (2 if r <= 7 else 1))
    else:
        R = 8 if r <= 5 else (4 if r <= 7 else 2)
    if R > 2 and tiles(n, H, W, 2 * R) < FEW_TILES:
        R = 2
    return ("bwrf32f_tiled", r, R, mode)


def group_frames(target_bytes, frame_bytes, n):
    """chunk_frames(..., spread = false) of dmc_capi.cu"""
    return max(1, min(target_bytes // frame_bytes, 65535, n))


def variants_chain(chain, params, n, H, W, dst, group_mb=GROUP_MB, lanes=1, overlap=False):
    """dmc_chain_batch on device memory: groups of group_mb / lanes MiB, each through run_chain.  The front stages write
    the context's scratch (aligned); the range filter writes dst, or the scratch when dst overlaps src."""
    mr, gr, mmr, br, th = params
    osize = {CHAIN_DISP8U: 1, CHAIN_DEPTH32F: 4}.get(chain, 2)
    group = group_frames((group_mb << 20) // lanes, H * W, n)
    out = []
    for f0 in range(0, n, group):
        nf = min(group, n - f0)
        out += [variant_median(mr, nf, H, W, 0) if mr else None, variant_gauss(gr, nf, H, W, 0), variant_minmax(mmr, nf, H, W, 0)]
        d = 0 if overlap else dst + f0 * H * W * osize
        if chain == CHAIN_DISP8U:
            out.append(variant_bwrf8u(br, th, nf, H, W, d))
        else:
            out.append(variant_bwrf32f(br, th, "u8" if chain == CHAIN_DISP32F else "u8disp", nf, H, W))
    return [v for v in out if v]


# ---------------------------------------------------------------------------------------------- reachable instantiations
def _table():
    t = set()
    for r in (1, 2):
        t |= {("median8u_p2", r, R, e) for R in (2, 16) for e in (False, True)}
    for r in range(3, 11):
        t |= {("median8u_bisect", r, 4, e) for e in (False, True)}
    t |= {("gauss8u_p4", 1, R, q) for R in (2, 8) for q in (False, True)}
    t |= {("gauss8u_p4", 2, R, q) for R in (2, 4) for q in (False, True)}
    for r in range(1, 6):
        t |= {("minmax8u_p2", r, R, e) for R in (4, 16) for e in (False, True)}
    for r in range(1, 11):
        full = 8 if r <= 3 else (4 if r <= 6 else (2 if r <= 8 else 1))
        # r = 1: no FLUSH, 5 taps * 255 (the largest 8-bit threshold) < 2048.  r >= 9: R = 1, no short variant
        flush = (False,) if r == 1 else (False, True)
        t |= {("bwrf8u_h2", r, R, f, e) for R in {full, min(full, 2)} for f in flush for e in (False, True)}
    for r in range(1, 8):
        # no size or store variants; r = 1: no FLUSH (5 * 255 < 2048)
        t |= {("bwrf8u_c3_h2", r, 4 if r <= 2 else (2 if r <= 5 else 1), f) for f in ((False,) if r == 1 else (False, True))}
    for r in range(1, 11):
        full = 8 if r <= 3 else (4 if r <= 5 else (2 if r <= 7 else 1))
        t |= {("bwrf32f_tiled", r, R, 0) for R in {full, min(full, 2)}}
        # MODE 1 / 2 stop at r = 9: the packed count holds at most 255 taps (253 at r = 9, 317 at r = 10)
        if r <= 9:
            full = 8 if r <= 5 else (4 if r <= 7 else 2)
            t |= {("bwrf32f_tiled", r, R, m) for R in {full, 2} for m in (1, 2)}
        # one tile height per radius: every R fits the 48 KB of static shared memory
        t.add(("bwrf32f_c3_tiled", r, 8 if r <= 3 else (4 if r <= 5 else (2 if r <= 7 else 1))))
    return t


TABLE = _table()


# ---------------------------------------------------------------------------------------------- the cases
class Case(NamedTuple):
    api: str            # "chain": dmc_chain_batch on device memory; "bwrf": binalyWeightedRangeFilter on one host image
    chain: int          # chain kind (api "chain")
    params: tuple       # (median_r, gaussian_r, minmax_r, brange_r, brange_th)
    load: str           # source type of api "bwrf": "u8", "u16", "s16", "f32"
    cn: int
    n: int
    H: int
    W: int
    src_off: int        # byte offsets of the batch in its device buffers (api "chain")
    dst_off: int

    def variants(self):
        if self.api == "chain":
            return variants_chain(self.chain, self.params, self.n, self.H, self.W, self.dst_off)
        r, th = self.params[3], self.params[4]
        if self.load == "u8":
            return [variant_bwrf8u(r, th, 1, self.H, self.W, 0, self.cn)]
        return [variant_bwrf32f(r, th, self.load, 1, self.H, self.W, self.cn)]

    def id(self):
        """e.g. minmax8u_p2-4-16-True-chain0-296x64x128-o16.2-0_0_4_0_0: the instantiation, then the call"""
        v = "-".join(str(x) for x in self.variants()[-1])
        return "%s-%s%s-%dx%dx%d-o%d.%d-%s" % (v, self.load if self.api == "bwrf" else "chain%d" % self.chain, "C3" if self.cn == 3 else "",
                                              self.n, self.H, self.W, self.src_off, self.dst_off, "_".join("%g" % x for x in self.params))


# Frame shapes: H is no multiple of any tile height except in (64, 128); W below 128, no multiple of 128, odd, and
# H = 1 with W = 2.  W = 256 and 128 with a 16-byte src take the 16-byte staging loads.
EVEN_W = [(70, 130), (33, 256), (1, 2), (50, 92), (64, 128)]
ODD_W = [(45, 67), (50, 97), (21, 131), (1, 3)]
QUAD_W = [(33, 256), (50, 92), (17, 124)]
NOT_QUAD_W = [(70, 130), (45, 67), (50, 97), (9, 2)]
SRC_OFFS = [0, 5, 16, 3]


def frames_for(full, n_tiles_per_frame):
    """the frame count at the boundary: the fewest frames that take the full variant, the most that take the short one"""
    return -(-FEW_TILES // n_tiles_per_frame) if full else max(1, (FEW_TILES - 1) // n_tiles_per_frame)


def _chain_cases():
    cases, k = [], 0

    def add(chain, params, shapes, full, tile_h, dst_odd=False, osize=1):
        nonlocal k
        H, W = shapes[k % len(shapes)]
        n = frames_for(full, tiles(1, H, W, tile_h)) if tile_h else 4
        dst_off = (1 if dst_odd else 0) + max(2, osize) * (k % 3)      # 16- and 32-bit outputs stay aligned
        cases.append(Case("chain", chain, params, "u8", 1, n, H, W, SRC_OFFS[k % len(SRC_OFFS)], dst_off))
        k += 1

    for r in range(1, 11):                                     # median alone
        for even in (True, False):
            for full in ((True, False) if r <= 2 else (True,)):
                add(CHAIN_DISP8U, (r, 0, 0, 0, 0), EVEN_W if even else ODD_W, full, 32 if r <= 2 else None)
    for gr in (1, 2):                                          # Gaussian alone (H = 1 takes the generic kernel)
        for quad in (True, False):
            for full in (True, False):
                add(CHAIN_DISP8U, (0, gr, 0, 0, 0), QUAD_W if quad else NOT_QUAD_W, full, 64)
    for r in range(1, 6):                                      # min-max alone
        for even in (True, False):
            for full in (True, False):
                add(CHAIN_DISP8U, (0, 0, r, 0, 0), EVEN_W if even else ODD_W, full, 64)
    for r in range(1, 11):                                     # 8-bit range filter alone: both sides of ntaps * th = 2048
        full_r = 8 if r <= 3 else (4 if r <= 6 else (2 if r <= 8 else 1))
        ths = [2048 // ntaps(r), 2048 // ntaps(r) + 1] if r > 1 else [255, 10]
        for th in ths:
            for even in (True, False):
                for full in ((True, False) if full_r > 2 else (True,)):
                    # byte stores from odd W and from an odd dst with an even W, in turn
                    odd_dst = not even and (k % 2 == 0)
                    add(CHAIN_DISP8U, (0, 0, 0, r, th), EVEN_W if even or odd_dst else ODD_W, full, 4 * full_r if full_r > 2 else None, dst_odd=odd_dst)
    add(CHAIN_DISP8U, (0, 0, 0, 3, 300.0), EVEN_W, True, 32)  # (uchar)300 = 44: the packed path, no FLUSH
    for r in range(1, 11):                                     # 32-bit range filter on the chain's 8-bit loads
        for chain, th, mode in ((CHAIN_DISP32F, 30.5, 1), (CHAIN_DEPTH32F, 65.0, 0)):
            if mode == 1 and r == 10:
                continue
            R = variant_bwrf32f(r, th, "u8" if mode else "u8disp", 10 ** 6, 64, 128)[2]
            for full in ((True, False) if R > 2 else (True,)):
                add(chain, (0, 0, 0, r, th), EVEN_W if k % 2 else ODD_W, full, 2 * R if R > 2 else None, osize=4 if chain == CHAIN_DEPTH32F else 2)
    return cases


BIG = [(520, 1100), (523, 1101)]      # at least 296 tiles at every full R (9 x 33 at R = 8)
SMALL = (37, 150)


def _bwrf_cases():
    cases = []
    for H, W in BIG:
        for load in ("u16", "s16", "f32"):
            for r in range(1, 11):
                for th in (37.5, 0.0, -1.0):                   # th < 0: the float path for integer sources too
                    cases.append(Case("bwrf", 0, (0, 0, 0, r, th), load, 1, 1, H, W, 0, 0))
        for r in range(1, 8):
            for th in sorted({10, 2048 // ntaps(r), 2048 // ntaps(r) + 1}):
                if (2 * r + 1) * th <= 2048 and th <= 255:
                    cases.append(Case("bwrf", 0, (0, 0, 0, r, th), "u8", 3, 1, H, W, 0, 0))
        for r in range(1, 11):
            cases.append(Case("bwrf", 0, (0, 0, 0, r, 30.5), "f32", 3, 1, H, W, 0, 0))
    for load in ("u16", "s16", "f32"):                         # the short variants
        for r in range(1, 8):
            cases.append(Case("bwrf", 0, (0, 0, 0, r, 37.5), load, 1, 1, SMALL[0], SMALL[1], 0, 0))
    return cases


CHAIN_CASES = _chain_cases()
BWRF_CASES = _bwrf_cases()
CASES = CHAIN_CASES + BWRF_CASES


def _mirror_image():
    """every instantiation the launchers can pick, by running the rules over a grid of inputs"""
    seen = set()
    shapes = [(64, 128), (64, 127), (1, 2)]
    for n in (1, 10 ** 5):
        for H, W in shapes:
            for dst in (0, 1):
                for r in range(0, 12):
                    seen |= {variant_median(r, n, H, W, dst) if r else None, variant_gauss(r, n, H, W, dst), variant_minmax(r, n, H, W, dst)}
                    for th in list(range(0, 256)) + [300.0, -1.0]:
                        seen |= {variant_bwrf8u(r, th, n, H, W, dst), variant_bwrf8u(r, th, n, H, W, dst, 3)}
                    for th in (-1.0, 0.0, 37.5, float("nan")):
                        for load in ("f32", "u16", "s16", "u8", "u8disp"):
                            seen |= {variant_bwrf32f(r, th, load, n, H, W), variant_bwrf32f(r, th, load, n, H, W, 3)}
    seen.discard(None)
    return seen


def test_table_is_what_the_rules_reach():
    mirror = _mirror_image()
    assert mirror == TABLE, "unreachable entries: %s; missing entries: %s" % (sorted(TABLE - mirror), sorted(mirror - TABLE))


def test_cases_reach_every_table_entry():
    reached = set()
    for c in CASES:
        v = c.variants()
        assert v and None not in v, c
        reached |= set(v)
    assert not TABLE - reached, "no case reaches %s" % sorted(TABLE - reached)
    assert reached <= TABLE, sorted(reached - TABLE)


# ---------------------------------------------------------------------------------------------- running the cases
@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)          # raises loudly without a GPU / without the built library
    return m


def _frames(seed, n, H, W):
    return np.stack([make_image(np.random.RandomState(seed + i), H, W) for i in range(n)])


def _guard(rs, H, W):
    return (rs.randint(0, 2, size=(H, W)) * 255).astype(np.uint8)


def _oracle_chain(port, chain, params, f):
    mr, gr, mmr, br, th = params
    if chain == CHAIN_DISP8U:
        return port.post_filter_set(f, mr, gr, mmr, br, th)
    if chain == CHAIN_DISP32F:
        return port.filter_disp8u_disp32f(f, mr, gr, mmr, br, th)
    return port.filter_disp8u_depth32f(f, FOCUS, BASELINE, AMP, mr, gr, mmr, br, th)


ODT = {CHAIN_DISP8U: np.uint8, CHAIN_DEPTH32F: np.float32, CHAIN_DEPTH16U: np.uint16, CHAIN_DISP32F: np.uint16}
MARK = 0xA5


def run_chain_device(dmc, ctx, frames, chain, params, src_off=0, dst_off=0, guards=None):
    """dmc_chain_batch on device memory.  src holds a guard frame before and after the batch; dst is a buffer of marker
    bytes with one frame of room before and after it.  -> (output frames, dst bytes outside the batch)"""
    import torch
    n, H, W = frames.shape
    fb, ob = H * W, H * W * np.dtype(ODT[chain]).itemsize
    g0, g1 = guards if guards is not None else (np.zeros((H, W), np.uint8),) * 2
    s = torch.zeros(src_off + (n + 2) * fb, dtype=torch.uint8, device="cuda")
    s[src_off:] = torch.from_numpy(np.concatenate([g0[None], frames, g1[None]]).reshape(-1)).cuda()
    d = torch.full((dst_off + (n + 2) * ob,), MARK, dtype=torch.uint8, device="cuda")
    p = dmc.filters.chain_params(chain, *params, focus=FOCUS, baseline=BASELINE, amp=AMP)
    torch.cuda.synchronize()
    ctx.chain_batch(s.data_ptr() + src_off + fb, d.data_ptr() + dst_off + ob, n, H, W, p, device=True)
    ctx.synchronize()
    out = d.cpu().numpy()
    got = out[dst_off + ob:dst_off + ob + n * ob].copy().view(ODT[chain]).reshape(n, H, W)
    return got, np.concatenate([out[:dst_off + ob], out[dst_off + ob + n * ob:]])


@pytest.mark.gpu
@pytest.mark.parametrize("case", CHAIN_CASES, ids=Case.id)
def test_chain_batch_variant(dmc, port, case):
    """one stage of the chain on a batch whose frame count puts it on the chosen side of the 2 x 148 tile boundary"""
    rs = np.random.RandomState(case.n * 7919 + case.H * 131 + case.W)
    frames = _frames(rs.randint(1 << 30), case.n, case.H, case.W)
    guards = (_guard(rs, case.H, case.W), _guard(rs, case.H, case.W))
    got, rest = run_chain_device(dmc, dmc.default_context(), frames, case.chain, case.params, case.src_off, case.dst_off, guards)
    assert (rest == MARK).all(), "%s: %d bytes outside the batch were written" % (case.variants(), int((rest != MARK).sum()))
    for i in range(case.n):
        assert_bits_equal(got[i], _oracle_chain(port, case.chain, case.params, frames[i]), "%s frame %d of %d" % (case.variants(), i, case.n))


@pytest.mark.gpu
@pytest.mark.parametrize("case", BWRF_CASES, ids=Case.id)
def test_single_image_variant(dmc, port, case):
    """16U / 16S / 32F / 8UC3 / 32FC3 sources, which the chain cannot feed, on images large enough for every full R"""
    dt = {"u8": np.uint8, "u16": np.uint16, "s16": np.int16, "f32": np.float32}[case.load]
    r, th = case.params[3], case.params[4]
    img = make_image(np.random.RandomState(case.H + 3 * r + case.cn), case.H, case.W, dt, case.cn)
    k = 2 * r + 1
    want = port.bwrf(img, k, k, th, FULL_KERNEL)
    got = dmc.binalyWeightedRangeFilter(img, None, (k, k), th, FULL_KERNEL)
    mask_undefined(got, want, k, k, case.W, FULL_KERNEL, dt, dmc)
    assert_bits_equal(got, want, str(case.variants()))


# ---------------------------------------------------------------------------------------------- groups and lanes
GROUP_SHAPE = (9, 130)               # 2 tiles per frame for every stage
GROUP_PARAMS = (2, 1, 3, 5, 10)


def _group_batch(port):
    H, W = GROUP_SHAPE
    # 1 MiB groups: 896 frames at lanes = 1, 448, 298 and 224 at 2, 3 and 4 lanes: full groups of >= 448 tiles, then a
    # last group of 3 or 7 frames (6 or 14 tiles)
    n = 2 * 896 + 3
    frames = _frames(500, n, H, W)
    want = np.stack([port.post_filter_set(f, *GROUP_PARAMS) for f in frames])
    return frames, want


@pytest.mark.gpu
def test_device_batch_groups_and_lanes(dmc, port, monkeypatch):
    """DMC_GROUP_MB = 1: many groups per call, the last one on the short variants; lanes = 1..4 run consecutive groups on
    different streams with their own scratch, and src / dst overlapping inside one allocation stage the output"""
    import torch
    H, W = GROUP_SHAPE
    frames, want = _group_batch(port)
    n = len(frames)
    ctx = dmc.default_context()
    monkeypatch.setenv("DMC_GROUP_MB", "1")
    outs = {}
    try:
        for lanes in (1, 2, 3, 4):
            v = variants_chain(CHAIN_DISP8U, GROUP_PARAMS, n, H, W, 0, group_mb=1, lanes=lanes)
            assert [x[2] for x in v[:4]] == [16, 8, 16, 4] and [x[2] for x in v[-4:]] == [2, 2, 4, 2], (lanes, v)
            ctx.set_lanes(lanes)
            got, rest = run_chain_device(dmc, ctx, frames, CHAIN_DISP8U, GROUP_PARAMS)
            assert (rest == MARK).all(), "lanes %d: bytes outside the batch were written" % lanes
            for i in range(n):
                assert_bits_equal(got[i], want[i], "lanes %d frame %d" % (lanes, i))
            outs[lanes] = got
            if lanes > 1:                                      # dst = src + half a frame: staged through the scratch
                buf = torch.zeros((n + 1) * H * W, dtype=torch.uint8, device="cuda")
                buf[:n * H * W] = torch.from_numpy(frames.reshape(-1)).cuda()
                p = dmc.filters.chain_params(CHAIN_DISP8U, *GROUP_PARAMS)
                torch.cuda.synchronize()
                ctx.chain_batch(buf.data_ptr(), buf.data_ptr() + H * W // 2, n, H, W, p, device=True)
                ctx.synchronize()
                ov = buf[H * W // 2:H * W // 2 + n * H * W].cpu().numpy().reshape(n, H, W)
                for i in range(n):
                    assert_bits_equal(ov[i], want[i], "overlapping src / dst, lanes %d frame %d" % (lanes, i))
    finally:
        ctx.set_lanes(1)
    for lanes in (2, 3, 4):
        assert_bits_equal(outs[lanes], outs[1], "lanes %d vs 1" % lanes)


@pytest.mark.gpu
def test_host_batch_cycles_slots(dmc, port, monkeypatch):
    """DMC_CHUNK_MB = 1: 11 chunks of 896 frames go through the four slots of the host-streamed path almost three times"""
    H, W = GROUP_SHAPE
    frames, want = _group_batch(port)
    reps = 5                                                   # chunk edges fall at other frames of the pattern each time
    big, wbig = np.concatenate([frames] * reps), np.concatenate([want] * reps)
    assert -(-len(big) // group_frames(1 << 20, H * W, len(big))) > 8
    monkeypatch.setenv("DMC_CHUNK_MB", "1")
    out = np.zeros_like(big)
    dmc.default_context().chain_batch(big, out, len(big), H, W, dmc.filters.chain_params(CHAIN_DISP8U, *GROUP_PARAMS), device=False)
    for i in range(len(big)):
        assert_bits_equal(out[i], wbig[i], "host batch frame %d" % i)


# ---------------------------------------------------------------------------------------------- the rules vs the kernels
KERNEL_RE = re.compile(r"\b(median8u_p2|median8u_bisect|gauss8u_p4|minmax8u_p2|bwrf8u_h2|bwrf8u_c3_h2|bwrf32f_tiled|bwrf32f_c3_tiled)_kernel<([^<>]*)>")


def _parse(name):
    """kernel name with its demangled template arguments -> the tuple the rules return (None for other kernels)"""
    m = KERNEL_RE.search(name)
    if not m:
        return None
    args = [a.strip() for a in m.group(2).split(",")]
    vals = [a == "true" if a in ("true", "false") else int(a.rstrip("uU")) for a in args]
    if m.group(1) == "median8u_p2":
        vals = [vals[0], vals[1], vals[5]]                      # RAD, R, EVEN (FNUM, FMOD, MINB: tuning constants)
    return (m.group(1),) + tuple(vals)


def _kernel_names(prof, path):
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    return [e["name"] for e in sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])]


@pytest.mark.gpu
def test_profiler_names(dmc, tmp_path):
    """one case per table entry: the kernels the profiler records, with their template arguments, are the ones the
    rules above predict, in launch order"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    x = torch.ones(1 << 16, device="cuda")
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        (x * 3).sum().item()
    assert _kernel_names(prof, tmp_path / "torch.json"), "the profiler recorded no CUDA kernel of a torch op: kernel names cannot be checked"

    chosen, seen = [], set()
    for c in CASES:
        if set(c.variants()) - seen:
            chosen.append(c)
            seen |= set(c.variants())
    assert seen == TABLE
    ctx = dmc.default_context()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        for c in chosen:
            if c.api == "chain":
                run_chain_device(dmc, ctx, np.zeros((c.n, c.H, c.W), np.uint8), c.chain, c.params, c.src_off, c.dst_off)
            else:
                dt = {"u8": np.uint8, "u16": np.uint16, "s16": np.int16, "f32": np.float32}[c.load]
                shape = (c.H, c.W) if c.cn == 1 else (c.H, c.W, 3)
                dmc.binalyWeightedRangeFilter(np.zeros(shape, dt), None, (2 * c.params[3] + 1,) * 2, c.params[4], FULL_KERNEL)
            ctx.synchronize()
    names = _kernel_names(prof, tmp_path / "cases.json")
    assert names, "the profiler recorded no CUDA kernel"
    got = [v for v in map(_parse, names) if v]
    want = [v for c in chosen for v in c.variants()]
    assert got, "no tiled kernel among the %d recorded kernels: %s" % (len(names), sorted(set(names))[:10])
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, "launch %d: the kernel ran %s, the rules predict %s" % (i, g, w)
    assert len(got) == len(want), "%d tiled kernels recorded, %d predicted" % (len(got), len(want))
