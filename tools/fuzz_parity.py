"""Randomised parity campaign (not part of the test suite; run on a GPU box when kernels change):
    python tools/fuzz_parity.py [seconds]
Draws shapes (biased to widths that are multiples of 16 / 4 / 2 and to sizes around the 128-px tile), radii, thresholds
and operators, and compares every result with the CPU oracle bit for bit."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import depthmapcompression_b200 as dmc
from oracle import oracle_py as O
import _float_edge_cases as E

budget = float(sys.argv[1]) if len(sys.argv) > 1 else 120.0
port = O.Port(); pfs = dmc.PostFilterSet(); rs = np.random.RandomState(int(os.environ.get("FUZZ_SEED", "12345")))
t0 = time.time(); n = 0; counts = {}


def image(H, W, cn=1):
    kind = rs.randint(3)
    shape = (H, W) if cn == 1 else (H, W, cn)
    if kind == 0: a = rs.randint(0, 256, size=shape)
    elif kind == 1:
        blk = rs.randint(1, 256, size=((H + 7) // 8, (W + 7) // 8) + (() if cn == 1 else (cn,)))
        a = np.kron(blk, np.ones((8, 8) + (() if cn == 1 else (1,))))[:H, :W] + rs.randint(-4, 5, size=shape)
    else:
        yy, xx = np.mgrid[0:H, 0:W]
        a = 128 + 100 * np.sin(xx / 17.0) * np.cos(yy / 11.0) + rs.randint(-2, 3, size=(H, W))
        if cn != 1: a = np.stack([a, 255 - a, (a * 3) % 256], axis=2)
    return np.ascontiguousarray(np.clip(a, 0, 255).astype(np.uint8))


def same(got, want, what):
    global n
    n += 1; counts[what.split()[0]] = counts.get(what.split()[0], 0) + 1
    if got.dtype.kind == "f":
        iv = np.uint32 if got.dtype == np.float32 else np.uint64
        ok = got.dtype == want.dtype and np.array_equal(got.view(iv)[~np.isnan(got)], want.view(iv)[~np.isnan(want)]) and np.array_equal(np.isnan(got), np.isnan(want))
    else:
        ok = np.array_equal(got, want)
    if not ok:
        bad = np.argwhere(got != want)
        print("MISMATCH", what, "shape", got.shape, "first", bad[:3].tolist(), "n", len(bad)); sys.exit(1)


while time.time() - t0 < budget:
    W = int(rs.choice([rs.randint(1, 40), 16 * rs.randint(1, 40), 4 * rs.randint(1, 150), 2 * rs.randint(1, 300), rs.randint(100, 300), 128 * rs.randint(1, 5) + rs.randint(-3, 4)]))
    H = int(rs.choice([rs.randint(1, 20), rs.randint(20, 140), 64 * rs.randint(1, 4) + rs.randint(-2, 3)]))
    W = max(W, 1); H = max(H, 1)
    a = image(H, W)
    op = rs.randint(13)
    if op == 0:
        k = int(rs.choice([3, 5, 7, 9, 13, 17, 21])); same(dmc.medianBlur(a, None, k) if hasattr(dmc, "medianBlur") else pfs(a, None, k // 2, 0, 0, 0, 0), port.post_filter_set(a, k // 2, 0, 0, 0, 0), "median k%d %dx%d" % (k, H, W))
    elif op == 1:
        r = int(rs.randint(1, 3)); same(pfs(a, None, 0, r, 0, 0, 0), port.post_filter_set(a, 0, r, 0, 0, 0), "gauss r%d %dx%d" % (r, H, W))
    elif op == 2:
        r = int(rs.randint(1, 6)); same(dmc.blurRemoveMinMax(a, None, r), port.blur_remove_minmax(a, r), "minmax r%d %dx%d" % (r, H, W))
    elif op == 3:
        r = int(rs.randint(1, 11)); th = int(rs.choice([0, 1, 5, 10, 25, 97, 140, 255])); k = 2 * r + 1
        same(dmc.binalyWeightedRangeFilter(a, None, (k, k), th, dmc.FULL_KERNEL), port.bwrf(a, k, k, th), "bwrf8u r%d th%d %dx%d" % (r, th, H, W))
    elif op == 4:
        c = image(H, W, 3); r = int(rs.randint(1, 8)); th = int(rs.choice([0, 10, 30, 140, 255])); k = 2 * r + 1
        same(dmc.binalyWeightedRangeFilter(c, None, (k, k), th, dmc.FULL_KERNEL), port.bwrf(c, k, k, th), "bwrf8uc3 r%d th%d %dx%d" % (r, th, H, W))
    elif op == 5:
        mr, gr, mmr, br, th = int(rs.randint(0, 3)), int(rs.randint(0, 3)), int(rs.randint(0, 4)), int(rs.randint(0, 6)), int(rs.randint(0, 40))
        b = np.maximum(a, 1)
        if rs.randint(2): same(pfs(b, None, mr, gr, mmr, br, th), port.post_filter_set(b, mr, gr, mmr, br, th), "chain8u %d,%d,%d,%d,%d %dx%d" % (mr, gr, mmr, br, th, H, W))
        else:
            if br == 5 and W % 4 == 0: br = 4      # the reference's own undefined read at r%8==5, cols%4==0 (masked in tests/)
            same(pfs.filterDisp8U2Depth32F(b, None, 75, 575, 2.6, mr, gr, mmr, br, th * 4.0), port.filter_disp8u_depth32f(b, 75, 575, 2.6, mr, gr, mmr, br, th * 4.0), "chain32f %d,%d,%d,%d,%d %dx%d" % (mr, gr, mmr, br, th, H, W))
    elif op == 6:
        k = int(rs.choice([3, 7, 13])); same(dmc.boundaryReconstructionFilter(a, None, (k, k), 1.0, 1.0, 1.0), port.brf(a, k, k, 1.0, 1.0, 1.0), "brf k%d %dx%d" % (k, H, W))
    elif op == 7:
        g = image(H, W, int(rs.choice([1, 3]))); r = int(rs.randint(1, 7)); th = int(rs.choice([0, 10, 30, 255])); k = 2 * r + 1
        same(dmc.jointBinalyWeightedRangeFilter(a, g, None, (k, k), th), port.joint_bwrf(a, g, k, k, th), "joint r%d th%d %dx%d" % (r, th, H, W))
    elif op == 8:       # boundary reconstruction filter on the other depths (hashed id table), non-square windows, weights
        dt = [np.uint16, np.int16, np.float32, np.float64][rs.randint(4)]
        lv = int(rs.choice([2, 5, 40, 300]))
        b = ((a.astype(np.int64) * lv // 256) * (37 if dt != np.float32 else 1)).astype(dt) if dt not in (np.float32, np.float64) else ((a.astype(np.int64) * lv // 256) * 0.37 - 11).astype(dt)
        kw, kh = int(rs.choice([3, 5, 7, 9, 13])), int(rs.choice([3, 5, 7, 13]))
        f, c, sp = [float(x) for x in rs.choice([0.0, 0.5, 1.0, 2.0], size=3)]
        same(dmc.boundaryReconstructionFilter(b, None, (kw, kh), f, c, sp), port.brf(b, kw, kh, f, c, sp), "brfT %s %dx%d k%dx%d" % (np.dtype(dt).name, H, W, kw, kh))
    elif op == 9:       # fused min-max -> boundary reconstruction (extension): oracle = composition of the two ports
        dt = [np.uint8, np.uint16, np.int16][rs.randint(3)]
        b = a.astype(dt) if dt == np.uint8 else (a.astype(np.int32) * 100 - (20000 if dt == np.int16 else 0)).astype(dt)
        r = int(rs.randint(0, 6)); k = int(rs.choice([3, 7, 9, 13]))
        same(dmc.minmaxBoundaryReconstructionFilter(b, None, r, (k, k), 1.0, 1.0, 1.0), port.brf(port.blur_remove_minmax(b, r), k, k, 1.0, 1.0, 1.0), "fused r%d k%d %s %dx%d" % (r, k, np.dtype(dt).name, H, W))
    elif op == 10:      # 32-bit range filter on 16-bit sources (integer mode up to radius 9, float mode at 10) and on floats
        dt = [np.uint16, np.int16, np.float32][rs.randint(3)]
        scale = int(rs.choice([1, 16, 257])); a = image(H, W, int(rs.choice([1, 3])))
        b = (a.astype(np.int32) * scale - (30000 if dt == np.int16 else 0)).clip(-32768, 65535).astype(dt) if dt != np.float32 else (a * 3.7).astype(np.float32)
        r = int(rs.randint(1, 11)); th = float(rs.choice([0, 0.5, 3, 10.9, 40, 160, 5000, 70000])); k = 2 * r + 1
        if dt == np.float32 and rs.randint(3) == 0:     # IEEE edge values, with thresholds that their distances meet exactly
            cases = E.CASES_C1 if a.ndim == 2 else E.CASES_C3
            case = cases[rs.randint(len(cases))]; b = case.image(H, W); ths = E.all_thresholds(case)
            th = float(ths[rs.randint(len(ths))])
        got = dmc.binalyWeightedRangeFilter(b, None, (k, k), th, dmc.FULL_KERNEL); want = port.bwrf(b, k, k, th)
        if r % 8 == 5 and W % 4 == 0: got[:, -1] = want[:, -1]      # the reference's own undefined read (masked in tests/ too)
        same(got, want, "bwrf32 %sC%d r%d th%s %dx%d" % (np.dtype(dt).name, a.size // (H * W), r, th, H, W))
    elif op == 11:      # blurRemoveMinMax on the wider types, NaN and zeros of both signs in the float images
        dt = [np.uint16, np.int16, np.float32, np.float64][rs.randint(4)]; cn = int(rs.choice([1, 3])); c = image(H, W, cn)
        if dt in (np.float32, np.float64):
            b = (c.astype(dt) - 128) * dt(0.5)
            sel = rs.rand(*b.shape); b[sel < 0.03] = np.nan; b[(sel >= 0.03) & (sel < 0.1)] = -0.0
        else:
            b = (c.astype(np.int32) * 257 - (32768 if dt == np.int16 else 0)).astype(dt)
        r = int(rs.randint(0, 11))
        same(dmc.blurRemoveMinMax(b, None, r), port.blur_remove_minmax(b, r), "minmaxT %sC%d r%d %dx%d" % (np.dtype(dt).name, cn, r, H, W))
    else:               # pinned host images (filtered in place over the host link)
        b = np.maximum(a, 1)
        if b.nbytes:
            pi = dmc.pinned_empty(b.shape, np.uint8); po = dmc.pinned_empty(b.shape, np.uint8); pi[:] = b
            same(pfs(pi, po, 1, 0, 1, 3, 10).copy(), port.post_filter_set(b, 1, 0, 1, 3, 10), "pinned %dx%d" % (H, W))
            dmc.pinned_free(pi); dmc.pinned_free(po)
print("fuzz ok: %d cases in %.0f s" % (n, time.time() - t0), counts)
