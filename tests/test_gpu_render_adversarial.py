"""The point-cloud render on adversarial geometry: projectImagefromXYZ (image, depth and pt), projectPointsSimple and
fillSmallHole of libdmc_b200.so must equal the port's literal serial loop (oracle/dmc_oracle.c, orc_project_image_serial)
bit for bit on scenes built from explicit points, where natural scenes never go:

  * dependency chains: point k's primary attempt fires only if point k-1's did not, because k-1's neighbour attempt
    z-tests k's pixel with a smaller z.  Along a row (left / right attempts), a column (up / down) and a diagonal (the
    down+right and up+left triples, whose last two attempts colour each other's pixel); one chain per row; up to
    125 000 links in one 3 x 250 001 image.  The renderer's fixed-point iteration can need one sweep per link, so these
    also bound its work (Context.kernel_launches);
  * z ties and extremes on one pixel, projection extremes (den = +-0, subnormal, >= 2^126, +-inf, NaN, negative;
    coordinates at the edges of cvttss2si and a neighbour at INT_MIN, which makes the right / down tests wrap on);
  * rcp_intel on every mantissa bucket at the exponents where its branches change;
  * the per-pixel sort on both sides of its insertion / heap switch and on 10^5 attempts;
  * fillSmallHole's blue / green tests and half-way quotients, tall and wide images;
  * frame batches (renderViewBatch, jpegViewRateDistortion) that put adversarial frames next to natural ones.

CPU part (no GPU): every generator builds what it claims, checked on the port alone.  GPU part: the library equals the
port, with exact division and, on Intel hosts, with the rcp table (the port executes the host's own RCPPS, whose table
is Intel's only on Intel CPUs: elsewhere those cases skip).

Non-finite z can never be drawn: z multiplies into every projected coordinate's numerator or denominator, so the
point projects to NaN (INT_MIN) whatever the camera.  The tie cases check exactly that.
"""
import numpy as np
import pytest

from _util import assert_bits_equal

F32 = np.float32
INT_MIN = -2 ** 31
I3, T0 = np.eye(3), np.zeros(3)


def sweep_cap(H, W):
    """sweeps before the serial finish (dmc_render.cu render_sweep_cap)"""
    return max(32, H * W // 1024)


def base_launches(H, W):
    """projectImagefromXYZ's kernels besides the sweeps: project, 3 x scan, sort, final sweep, resolve, and count and fill
    once per 65535 interior rows"""
    chunks = -(-(H - 2) // 65535) if H > 2 and W > 2 else 0
    return 7 + 2 * chunks


def intel_host():
    try:
        return "GenuineIntel" in open("/proc/cpuinfo").read()
    except Exception:
        return False


# ---- a restatement of the attempt rules, for the CPU checks ----------------------------------------------------------
def f2i(v):
    """(int)v as cvttss2si does it, elementwise: out of range / NaN -> INT_MIN"""
    v = np.asarray(v, F32)
    with np.errstate(invalid="ignore"):
        ok = (v > F32(-2147483904.0)) & (v < F32(2147483648.0))
    out = np.full(v.shape, INT_MIN, np.int64)
    out[ok] = np.trunc(v[ok]).astype(np.int64)
    return out


def sub_wrap(a, b):
    return ((np.asarray(a, np.int64) - b + 2 ** 31) % 2 ** 32) - 2 ** 31


def attempt_flags(pt, H, W):
    """-> dict of [H-2, W-2] bool maps over the interior points: on (primary attempt), right, down, up, left (isSub)"""
    px, py = f2i(pt[:, 0]).reshape(H, W), f2i(pt[:, 1]).reshape(H, W)
    x, y = px[1:-1, 1:-1], py[1:-1, 1:-1]
    on = (x >= 1) & (x < W - 1) & (y >= 1) & (y < H - 1)
    return {"on": on, "right": on & (sub_wrap(px[1:-1, 2:], x) > 1), "down": on & (sub_wrap(py[2:, 1:-1], y) > 1),
            "up": on & (sub_wrap(py[:-2, 1:-1], y) < -1), "left": on & (sub_wrap(px[1:-1, :-2], x) < -1), "x": x, "y": y}


def colours(H, W, seed=0):
    rs = np.random.RandomState(seed)
    return rs.randint(1, 256, (H, W, 3)).astype(np.uint8)


# ---- generators ----------------------------------------------------------------------------------------------------
# Every scene is (H, W, xyz [H*W, 3], R, t, K) plus what it claims.  Most use K = R = I and t = 0, so a point (x, y, z)
# projects to (x / z, y / z): the grid scene puts every point on its own pixel centre, (i + 0.5, j + 0.5).
def grid_xyz(H, W):
    xyz = np.ones((H, W, 3), F32)
    xyz[..., 0] = np.arange(W)[None, :] + 0.5
    xyz[..., 1] = np.arange(H)[:, None] + 0.5
    return xyz


def link_z(k):
    return F32(1.0 + k / 1024.0)


def row_chains(L, leftward, H=3):
    """In every interior row, L links at the odd columns (link k at column 2k + 1) between helpers that project far
    off-screen to the left (leftward) or right, so every link also attempts its left (right) neighbour pixel.  Leftward,
    link k targets column W-2-k and its left attempt column W-3-k, link k+1's target; rightward link k targets column
    1+k.  z grows along the chain, so the serial splat fires links 0, 2, 4, ...  -> H, W, xyz, links [(row, col)],
    targets [(row, col)]"""
    W = 2 * L + 1
    xyz = grid_xyz(H, W)
    xyz[1:-1, :, 0] = -1e6 if leftward else 1e6
    links, targets = [], []
    for j in range(1, H - 1):
        for k in range(L):
            u = W - 2 - k if leftward else 1 + k
            z = link_z(k)
            xyz[j, 2 * k + 1] = ((u + 0.5) * z, (j + 0.5) * z, z)
            links.append((j, 2 * k + 1)); targets.append((j, u))
    return H, W, xyz.reshape(-1, 3), links, targets


def column_chain(L, upward):
    """row_chains turned on its side: a (2L+1) x 3 image, links at the odd rows of column 1, helpers far up (down)."""
    H, W = 2 * L + 1, 3
    xyz = grid_xyz(H, W)
    xyz[:, 1, 1] = -1e6 if upward else 1e6
    links, targets = [], []
    for k in range(L):
        v = H - 2 - k if upward else 1 + k
        z = link_z(k)
        xyz[2 * k + 1, 1] = (1.5 * z, (v + 0.5) * z, z)
        links.append((2 * k + 1, 1)); targets.append((v, 1))
    return H, W, xyz.reshape(-1, 3), links, targets


def diagonal_chain(L, down_right):
    """Links at the (odd row, odd column) points in raster order, every other point a helper far down-right (up-left), so
    each link makes the down+right (up+left) triple; the triple's diagonal attempt z-tests the next link's target: link
    k targets (1+k, 1+k) (or (N-2-k, N-2-k))."""
    N = L + 3
    while ((N - 1) // 2) ** 2 < L:
        N += 1
    xyz = grid_xyz(N, N)
    far = 1e6 if down_right else -1e6
    xyz[..., 0] = far; xyz[..., 1] = far
    slots = [(j, i) for j in range(1, N - 1, 2) for i in range(1, N - 1, 2)][:L]
    targets = []
    for k, (j, i) in enumerate(slots):
        u = 1 + k if down_right else N - 2 - k
        z = link_z(k)
        xyz[j, i] = ((u + 0.5) * z, (u + 0.5) * z, z)
        targets.append((u, u))
    return N, N, xyz.reshape(-1, 3), slots, targets


# One pixel, many points: R maps (x, y, z) to (x, 1.5 y, y), so every point (3.5, 1, z) of a 3-row image projects to
# pixel (3, 1) whatever its z, as long as z is finite.
R_TIE = np.array([[1.0, 0, 0], [0, 1.5, 0], [0, 1.0, 0]])
TIES = {
    "equal": [5.0, 5.0, 5.0, 7.0],
    "zero_then_negzero": [0.0, -0.0, 1.0],
    "negzero_then_zero": [-0.0, 0.0, 1.0],
    "z10000": [10000.0, float(np.nextafter(F32(10000), F32(0))), 10000.0],
    "nonfinite": [float("nan"), 3.0, float("-inf"), 2.0, float("inf"), 1.0],
    "negative": [2.0, -1.0, -1.0, -5.0, 0.0],
}


def tie_scene(zs, pad_to=5):
    zs = list(zs) + [20000.0] * max(0, pad_to - 2 - len(zs))           # padding points are never drawn (10000 > 20000 fails)
    H, W = 3, len(zs) + 2
    xyz = np.zeros((H, W, 3), F32)
    xyz[..., 0], xyz[..., 1], xyz[..., 2] = 3.5, 1.0, 1.0
    xyz[1, 1:-1, 2] = np.array(zs, F32)
    return H, W, xyz.reshape(-1, 3)


def tie_expect(zs):
    """index of the drawn point that remains (first strict minimum below 10000 of the finite z: a non-finite z projects
    off-screen), or None"""
    cur, win = F32(10000), None
    for k, z in enumerate(np.array(zs, F32)):
        if np.isfinite(z) and cur > z:
            cur, win = z, k
    return win


DEN_SPECIAL = {"+0": 0.0, "-0": -0.0, "subnormal": 1e-40, "-subnormal": -1e-40, "2^126": 2.0 ** 126, "1.5*2^127": 1.5 * 2.0 ** 127,
               "+inf": float("inf"), "-inf": float("-inf"), "nan": float("nan"), "negative": -2.0}
COORD_EDGE = {"-2147483904": -2147483904.0, "-2^31": -2.0 ** 31, "2^31": 2.0 ** 31, "nan": float("nan"),
              "below 2^31": 2147483520.0, "above -2147483904": -2147483520.0}


def zoo(H, W, seed):
    """Random points from a palette: 60 % on-screen (targets crowded into a few pixels, z from a small set with ties and
    negatives), 20 % with a special denominator (z), 20 % with a coordinate at an edge of cvttss2si (z = 1)."""
    rs = np.random.RandomState(seed)
    xyz = np.zeros((H * W, 3), F32)
    zset = np.array([1.0, 2.0, 0.5, -2.0, 3.0, 3.0, 7.5], F32)
    dens, edges = list(DEN_SPECIAL.values()), list(COORD_EDGE.values())
    for p in range(H * W):
        r = rs.rand()
        if r < 0.6:
            z = zset[rs.randint(len(zset))]
            u, v = rs.randint(1, max(2, min(W - 1, 5))), rs.randint(1, max(2, min(H - 1, 4)))
            xyz[p] = ((u + 0.5) * z, (v + 0.5) * z, z)
        elif r < 0.8:
            with np.errstate(over="ignore"):                # x * 2^127 may round to inf: one more special
                xyz[p] = (rs.uniform(-3, 3) * 2.0 ** rs.choice([0, 126, 127]), rs.uniform(1, 3), dens[rs.randint(len(dens))])
        else:
            e = edges[rs.randint(len(edges))]
            xyz[p] = (e, rs.uniform(1, 3), 1.0) if rs.rand() < 0.5 else (rs.uniform(1, 3), e, 1.0)
    # make sure each special shows up at least once, and a neighbour at INT_MIN beside an on-screen point
    for k, d in enumerate(dens):
        xyz[k] = (3.0, 2.0, d)
    for k, e in enumerate(edges):
        xyz[len(dens) + 2 * k] = (e, 1.5, 1.0); xyz[len(dens) + 2 * k + 1] = (1.5, e, 1.0)
    j = H // 2
    xyz[j * W + 1] = (2.5, 1.5, 1.0)
    xyz[j * W + 2] = (float("nan"), 1.5, 1.0)
    xyz[(j + 1) * W + 1] = (1.5, float("nan"), 1.0)
    return xyz


def rcp_dens():
    """Every one of the 2048 mantissa buckets of rcp_intel, at its first, last and a middle mantissa, for biased exponents
    1, 2, 126-128 and 251-254 and both signs."""
    m = np.arange(2048, dtype=np.uint32) << 12
    ms = np.concatenate([m, m | 0xfff, m | 0x7a5])
    bits = [(s << 31) | (e << 23) | ms for s in (0, 1) for e in (1, 2, 126, 127, 128, 251, 252, 253, 254)]
    return np.concatenate(bits).astype(np.uint32).view(F32)


def rcp_scene(dens):
    """projectPointsSimple with K = R = I, t = 0 and the point (1, 0, den): pt.x is the reciprocal of den."""
    xyz = np.zeros((len(dens), 3), F32)
    xyz[:, 0] = 1.0; xyz[:, 2] = dens
    return xyz


def hole_image(H, W, seed):
    """Small channel values, so holes (green 0) and non-neighbours (blue 0) are frequent and quotients often k + 0.5."""
    rs = np.random.RandomState(seed)
    img = rs.choice(np.array([0, 0, 1, 2, 3, 4, 5, 200, 255], np.uint8), (H, W, 3))
    return np.ascontiguousarray(img)


def hole_quotients(img):
    """-> (holes with blue != 0, points with blue == 0 and green != 0, quotients exactly k + 0.5 with k even / odd)"""
    H, W = img.shape[:2]
    s = img.astype(np.int64)
    c = s[1:-1, 1:-1]
    hole = c[..., 1] == 0
    cnt = np.zeros((H - 2, W - 2), np.int64); sums = np.zeros((H - 2, W - 2, 3), np.int64)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            if dy or dx:
                q = s[1 + dy:H - 1 + dy, 1 + dx:W - 1 + dx]
                nz = q[..., 0] != 0
                cnt += nz; sums += q * nz[..., None]
    m = hole & (cnt > 0)
    twice = 2 * sums[m]; cn = cnt[m][:, None]
    half = (twice % cn == 0) & ((twice // cn) % 2 == 1)
    k = (twice // cn) // 2
    return (int((hole & (c[..., 0] != 0)).sum()), int(((c[..., 0] == 0) & (c[..., 1] != 0)).sum()),
            int((half & (k % 2 == 0)).sum()), int((half & (k % 2 == 1)).sum()))


CHAIN_LENGTHS = [1, 2, 31, 32, 33, 255, 256, 257, 2000]


# A chain inside a frame batch: renderViewBatch reprojects 32F depth (reprojectXYZ, focal length VIEW_F) and renders it
# with the camera R = I, t = (VIEW_TX, 0, 0) and view_intrinsics.  A point of column i and row j at depth Z > 0 then lands
# near (i + 0.5 + VIEW_F * VIEW_TX / Z, j + 0.5): every point stays in its own row, so rows make no up / down attempts
# and do not interact.
VIEW_F, VIEW_TX = 100.0, 1.0


def view_intrinsics(H, W):
    K = np.eye(3) * VIEW_F
    K[0, 2], K[1, 2], K[2, 2] = (W - 1) * 0.5 + 0.5, (H - 1) * 0.5 + 0.5, 1.0      # pixel centres half a pixel off the borders
    return K


def view_chain_depth(natural, L):
    """`natural` with row 1 replaced by a rightward chain of L links: link k at column 2k + 1 with Z = f tx / (L - k)
    lands on column L + 1 + k, and the points between, at Z = 1e-4, land far right, so every link attempts its right
    neighbour pixel, the next link's target.  Z grows along the chain, so the serial splat fires links 0, 2, 4, ...
    -> depth, links [(row, col)], targets [(row, col)]"""
    H, W = natural.shape
    assert W >= 2 * L + 2
    d = natural.astype(F32).copy()
    d[1, :] = 1e-4
    links, targets = [], []
    for k in range(L):
        d[1, 2 * k + 1] = F32(VIEW_F * VIEW_TX / (L - k))
        links.append((1, 2 * k + 1)); targets.append((1, L + 1 + k))
    return d, links, targets


VIEW_CHAINS = {1: 100, 3: 60}               # frame index -> links, between natural frames


def view_chain_batch():
    """Five 24 x 202 32F frames: natural depth at 0, 2 and 4, chains of 100 and 60 links at 1 and 3."""
    from oracle.oracle_py import Port, synth_disp
    port = Port()
    H, W = 24, 202
    frames, chains = [], {}
    for i in range(5):
        natural = port.filter_disp8u_depth32f(synth_disp(H, W, 40 + i), 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0)
        if i in VIEW_CHAINS:
            d, links, targets = view_chain_depth(natural, VIEW_CHAINS[i])
            chains[i] = (links, targets)
        else:
            d = natural
        frames.append(d)
    return np.stack(frames), chains


# ---- CPU: the generators build what they claim ---------------------------------------------------------------------
def fired_links(port, H, W, xyz, links, targets):
    """Which links the serial splat fired (exact division): a link fired iff its target keeps its own z.  (The only
    other attempt on a target is the previous link's, with a smaller z.)"""
    col = colours(H, W)
    _, depth = port.project_image(col, xyz, I3, T0, I3, True, rcp=False)
    z = xyz.reshape(H, W, 3)[..., 2]
    return np.array([depth[t] == z[l] for l, t in zip(links, targets)])


@pytest.mark.parametrize("L", CHAIN_LENGTHS)
@pytest.mark.parametrize("kind", ["left", "right", "up", "down", "down_right", "up_left"])
def test_chains_alternate(port, kind, L):
    if kind in ("left", "right"):
        H, W, xyz, links, targets = row_chains(L, kind == "left")
    elif kind in ("up", "down"):
        H, W, xyz, links, targets = column_chain(L, kind == "up")
    else:
        if L > 300:
            pytest.skip("diagonal chains are square images: kept to a few hundred links")
        H, W, xyz, links, targets = diagonal_chain(L, kind == "down_right")
    pt = port.project_points(xyz, I3, T0, I3, rcp=False)
    fl = attempt_flags(pt, H, W)
    attempt = {"left": "left", "right": "right", "up": "up", "down": "down"}
    for (j, i), tgt in zip(links, targets):
        assert fl["on"][j - 1, i - 1] and (fl["y"][j - 1, i - 1], fl["x"][j - 1, i - 1]) == tgt, (kind, j, i)
        if kind in attempt:
            assert fl[attempt[kind]][j - 1, i - 1], (kind, j, i)
        else:
            a, b = ("down", "right") if kind == "down_right" else ("up", "left")
            assert fl[a][j - 1, i - 1] and fl[b][j - 1, i - 1], (kind, j, i)
    assert fl["on"].sum() == len(links)                     # helpers make no attempts
    fired = fired_links(port, H, W, xyz, links, targets)
    assert np.array_equal(fired, np.arange(len(links)) % 2 == 0), kind


def test_multi_row_and_long_chains_alternate(port):
    H, W, xyz, links, targets = row_chains(100, True, H=7)
    assert len({t[0] for t in targets}) == 5
    fired = fired_links(port, H, W, xyz, links, targets).reshape(5, 100)
    assert np.all(fired == (np.arange(100) % 2 == 0))
    H, W, xyz, links, targets = long_chain()
    assert (H, W, len(links)) == (3, 250001, 125000)
    fired = fired_links(port, H, W, xyz, links, targets)
    assert np.array_equal(fired, np.arange(len(links)) % 2 == 0)


def long_chain():
    return row_chains(125000, True)


def test_view_chains_alternate(port):
    depth, chains = view_chain_batch()
    _, H, W = depth.shape
    K, t = view_intrinsics(H, W), np.array([VIEW_TX, 0.0, 0.0])
    for i, (links, targets) in chains.items():
        xyz = port.reproject_xyz(depth[i], VIEW_F)
        for rcp in (False, True):
            fl = attempt_flags(port.project_points(xyz, I3, t, K, rcp=rcp), H, W)
            assert not (fl["up"] | fl["down"]).any(), (i, rcp)
            for (j, c), tgt in zip(links, targets):
                assert fl["on"][j - 1, c - 1] and fl["right"][j - 1, c - 1], (i, rcp, c)
                assert (fl["y"][j - 1, c - 1], fl["x"][j - 1, c - 1]) == tgt, (i, rcp, c)
            assert fl["on"][0].sum() == len(links)            # the points between the links stay off-screen
        _, zbuf = port.project_image(colours(H, W), xyz, I3, t, K, True, rcp=False)
        fired = np.array([zbuf[tg] == depth[i][l] for l, tg in zip(links, targets)])
        assert np.array_equal(fired, np.arange(len(links)) % 2 == 0), i


def test_ties_land_on_one_pixel(port):
    for name, zs in TIES.items():
        H, W, xyz = tie_scene(zs)
        for rcp in (False, True):
            pt = port.project_points(xyz, R_TIE, T0, I3, rcp=rcp)
            px, py = f2i(pt[:, 0]).reshape(H, W), f2i(pt[:, 1]).reshape(H, W)
            zrow = xyz.reshape(H, W, 3)[1, 1:-1, 2]
            fin = np.isfinite(zrow)
            assert np.all(px[1, 1:-1][fin] == 3) and np.all(py[1, 1:-1][fin] == 1), (name, rcp)
            assert np.all(px[1, 1:-1][~fin] == INT_MIN), (name, rcp)             # non-finite z: never on screen
        col = colours(H, W, 5)
        dest, depth = port.project_image(col, xyz, R_TIE, T0, I3, True, rcp=False)
        win = tie_expect(zs)
        if win is None:
            assert depth[1, 3] == 10000 and not dest[1, 3].any(), name
        else:
            assert np.array_equal(dest[1, 3], col[1, 1 + win]), name
            assert depth[1, 3].view(np.uint32) == F32(zs[win]).view(np.uint32), name
    assert tie_expect(TIES["equal"]) == 0 and tie_expect(TIES["zero_then_negzero"]) == 0 and tie_expect(TIES["negzero_then_zero"]) == 0
    assert tie_expect(TIES["z10000"]) == 1 and tie_expect(TIES["nonfinite"]) == 5 and tie_expect(TIES["negative"]) == 3


ZOO_SHAPES = ((9, 12), (5, 13), (6, 11), (7, 9))


def test_zoo_reaches_every_edge(port):
    assert {(H * W) % 4 for H, W in ZOO_SHAPES} == {0, 1, 2, 3}                  # the scalar tail takes 0..3 points
    for H, W in ZOO_SHAPES:
        xyz = zoo(H, W, H * W)
        z = xyz[:, 2]
        for name, d in DEN_SPECIAL.items():
            hit = np.isnan(z) if np.isnan(d) else (z == d) & (np.signbit(z) == np.signbit(d))
            assert hit.any(), name
        pt = port.project_points(xyz, I3, T0, I3, rcp=False)
        for name, e in COORD_EDGE.items():
            for c in (0, 1):
                hit = np.isnan(pt[:, c]) if np.isnan(e) else pt[:, c] == F32(e)
                assert hit.any(), (name, c)
        fl = attempt_flags(pt, H, W)
        px, py = f2i(pt[:, 0]).reshape(H, W), f2i(pt[:, 1]).reshape(H, W)
        wrap_r = fl["right"] & (px[1:-1, 2:] == INT_MIN)
        wrap_d = fl["down"] & (py[2:, 1:-1] == INT_MIN)
        assert wrap_r.any() and wrap_d.any() and (wrap_r & wrap_d).any(), (H, W)
        assert (fl["on"] & (xyz.reshape(H, W, 3)[1:-1, 1:-1, 2] < 0)).any()        # points behind the camera are drawn
        for k in ("up", "left"):
            assert fl[k].any(), k


def test_rcp_scene_is_the_reciprocal(port):
    dens = rcp_dens()
    b = dens.view(np.uint32)
    assert len(dens) % 4 == 0                               # every point takes the SIMD body's reciprocal
    for s in (0, 1):
        for e in (1, 2, 126, 127, 128, 251, 252, 253, 254):
            sel = ((b >> 31) == s) & (((b >> 23) & 0xff) == e)
            assert np.array_equal(np.unique((b[sel] >> 12) & 0x7ff), np.arange(2048)), (s, e)
    pt = port.project_points(rcp_scene(dens), I3, T0, I3, rcp=False)
    with np.errstate(over="ignore", divide="ignore"):
        assert_bits_equal(pt[:, 0], F32(1) / dens, "exact pt.x == 1 / den")


def test_sort_scenes_count_attempts(port):
    for m in (48, 49):
        H, W, xyz = tie_scene(np.random.RandomState(m).choice([1.0, 2.0, 3.0], m))
        fl = attempt_flags(port.project_points(xyz, R_TIE, T0, I3, rcp=False), H, W)
        assert fl["on"].sum() == m and not (fl["right"] | fl["left"] | fl["up"] | fl["down"]).any()
    H, W, xyz = crowd_scene()
    fl = attempt_flags(port.project_points(xyz, I3, T0, I3, rcp=False), H, W)
    assert fl["on"].all() and np.all(fl["x"] == 3) and np.all(fl["y"] == 3) and fl["on"].sum() > 100000


def crowd_scene(N=320, seed=9):
    """N x N points with z in [1, 100) that all project to pixel (3, 3): (N-2)^2 > 10^5 attempts on one pixel."""
    rs = np.random.RandomState(seed)
    z = rs.uniform(1, 100, N * N).astype(F32)
    z[::7] = z[0]                                           # ties
    return N, N, np.stack([F32(3.5) * z, F32(3.5) * z, z], -1).astype(F32)


HOLE_SHAPES = [(40, 50), (3, 3000), (3000, 3), (70001, 3), (3, 70001)]


def test_hole_images_reach_every_case():
    for H, W in HOLE_SHAPES:
        hb, bg, even, odd = hole_quotients(hole_image(H, W, H + W))
        assert hb > 0 and bg > 0 and even > 0 and odd > 0, (H, W)


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


@pytest.fixture(params=["exact", "rcp"])
def exact(request):
    if request.param == "rcp" and not intel_host():
        pytest.skip("the port's RCPPS follows the host CPU; the library carries Intel's table: needs an Intel host")
    return request.param == "exact"


def render_equals_port(dmc, port, H, W, xyz, R, t, K, exact, what, subs=(False, True), seed=0):
    """-> kernel launches of the last call"""
    col = colours(H, W, seed)
    ctx = dmc.default_context()
    want_pt = port.project_points(xyz, R, t, K, rcp=not exact)
    n = 0
    for sub in subs:
        want, wz = port.project_image(col, xyz, R, t, K, sub, rcp=not exact)
        n0 = ctx.kernel_launches
        got, gz, gpt = dmc.projectImagefromXYZ(col, None, xyz, R, t, K, isSub=sub, want_depth=True, exact_divide=exact)
        n = ctx.kernel_launches - n0
        tag = "%s isSub=%d exact=%d" % (what, sub, exact)
        assert_bits_equal(gpt, want_pt, tag + " pt")
        assert_bits_equal(gz, wz, tag + " depth")
        assert_bits_equal(got, want, tag + " image")
        base = base_launches(H, W)
        assert n == base if not sub else base < n <= base + sweep_cap(H, W) + 1, (tag, n)
    return n


@pytest.mark.gpu
@pytest.mark.parametrize("L", CHAIN_LENGTHS)
@pytest.mark.parametrize("leftward", [True, False], ids=["left", "right"])
def test_gpu_row_chains(dmc, port, exact, leftward, L):
    H, W, xyz, _, _ = row_chains(L, leftward)
    render_equals_port(dmc, port, H, W, xyz, I3, T0, I3, exact, "row chain L=%d left=%d" % (L, leftward))


@pytest.mark.gpu
def test_gpu_multi_row_column_and_diagonal_chains(dmc, port, exact):
    H, W, xyz, _, _ = row_chains(300, True, H=9)
    render_equals_port(dmc, port, H, W, xyz, I3, T0, I3, exact, "one chain per row")
    for L in (1, 2, 33, 257, 2000):
        for up in (True, False):
            H, W, xyz, _, _ = column_chain(L, up)
            render_equals_port(dmc, port, H, W, xyz, I3, T0, I3, exact, "column chain L=%d up=%d" % (L, up))
    for L in (1, 2, 33, 257):
        for dr in (True, False):
            H, W, xyz, _, _ = diagonal_chain(L, dr)
            render_equals_port(dmc, port, H, W, xyz, I3, T0, I3, exact, "diagonal chain L=%d down_right=%d" % (L, dr))


@pytest.mark.gpu
def test_gpu_long_chain(dmc, port):
    """125 000 links: the fixed point alone would need about one sweep (a launch and a host round trip) per link."""
    H, W, xyz, _, _ = long_chain()
    col = colours(H, W)
    want, wz = port.project_image(col, xyz, I3, T0, I3, True, rcp=False)
    ctx = dmc.default_context()
    n0 = ctx.kernel_launches
    got, gz, _ = dmc.projectImagefromXYZ(col, None, xyz, I3, T0, I3, isSub=True, want_depth=True, exact_divide=True)
    n = ctx.kernel_launches - n0
    assert_bits_equal(gz, wz, "long chain depth")
    assert_bits_equal(got, want, "long chain image")
    assert n == base_launches(H, W) + sweep_cap(H, W) + 1, n               # the capped sweeps, then the serial finish


@pytest.mark.gpu
def test_gpu_natural_scenes_settle_within_the_cap(dmc, port):
    """The serial finish is for adversarial input only: natural views settle in a few sweeps."""
    from oracle.oracle_py import synth_disp
    from test_pointcloud import VIEWS
    H, W = 240, 320
    d32 = port.filter_disp8u_depth32f(synth_disp(H, W, 5), 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0)
    xyz = port.reproject_xyz(d32, 300.0)
    K = np.eye(3) * 300.0; K[0, 2] = (W - 1) * 0.5; K[1, 2] = (H - 1) * 0.5; K[2, 2] = 1.0
    for name, R, t in VIEWS:
        n = render_equals_port(dmc, port, H, W, xyz, R, t, K, True, name, subs=(True,))
        assert n < base_launches(H, W) + sweep_cap(H, W), (name, n)


@pytest.mark.gpu
def test_gpu_ties_and_extremes_on_one_pixel(dmc, port, exact):
    for name, zs in TIES.items():
        H, W, xyz = tie_scene(zs)
        render_equals_port(dmc, port, H, W, xyz, R_TIE, T0, I3, exact, "tie " + name)


@pytest.mark.gpu
def test_gpu_projection_extremes(dmc, port, exact):
    for H, W in ZOO_SHAPES + ((2, 9), (9, 2)):
        xyz = zoo(H, W, H * W) if H > 2 and W > 2 else np.full((H * W, 3), np.nan, F32)
        render_equals_port(dmc, port, H, W, xyz, I3, T0, I3, exact, "zoo %dx%d" % (H, W), seed=H)
        assert_bits_equal(dmc.projectPointsSimple(xyz, I3, T0, I3, exact_divide=exact), port.project_points(xyz, I3, T0, I3, rcp=not exact), "zoo pt")
    for seed in range(4):                                   # larger zoos, tall and wide
        for H, W in ((31, 45), (70001, 3), (3, 5003)):
            if H * W > 100000 and seed:
                continue
            render_equals_port(dmc, port, H, W, zoo(H, W, 100 + seed), I3, T0, I3, exact, "zoo %dx%d seed %d" % (H, W, seed), seed=seed)


@pytest.mark.gpu
def test_gpu_rcp_intel_every_bucket(dmc, port):
    if not intel_host():
        pytest.skip("the port's RCPPS follows the host CPU; the library carries Intel's table: needs an Intel host")
    dens = rcp_dens()
    xyz = rcp_scene(dens)
    assert_bits_equal(dmc.projectPointsSimple(xyz, I3, T0, I3), port.project_points(xyz, I3, T0, I3, rcp=True), "rcp_intel buckets")
    special = np.array(list(DEN_SPECIAL.values()) + [2.0 ** -126, 2.0 ** -127, -2.0 ** 127, 3.4e38, 1.0, -1.0], F32)
    xyz = rcp_scene(np.concatenate([special, special[:2]]))           # a multiple of 4: all through the table
    assert_bits_equal(dmc.projectPointsSimple(xyz, I3, T0, I3), port.project_points(xyz, I3, T0, I3, rcp=True), "rcp_intel specials")


@pytest.mark.gpu
def test_gpu_sort_paths(dmc, port, exact):
    for m in (47, 48, 49, 50):
        H, W, xyz = tie_scene(np.random.RandomState(m).choice([1.0, 2.0, 3.0], m))
        render_equals_port(dmc, port, H, W, xyz, R_TIE, T0, I3, exact, "%d attempts on one pixel" % m)
    H, W, xyz = crowd_scene()                                # one heap sort of 10^5 entries, and a few sweeps over them
    render_equals_port(dmc, port, H, W, xyz, I3, T0, I3, exact, "crowd", subs=(False, True))


@pytest.mark.gpu
def test_gpu_fill_small_hole(dmc, port):
    for H, W in HOLE_SHAPES:
        img = hole_image(H, W, H + W)
        want = port.fill_small_hole(img)
        assert_bits_equal(dmc.fillSmallHole(img.copy()), want, "%dx%d in place" % (H, W))
        canvas = np.full_like(img, 37)
        assert_bits_equal(dmc.fillSmallHole(img, canvas.copy()), port.fill_small_hole(img, canvas), "%dx%d into a canvas" % (H, W))


# -- batches ---------------------------------------------------------------------------------------------------------
MIRROR = np.diag([-1.0, -1.0, 1.0])


def batch_cameras():
    """identity, the mirrored camera (later raster points land further left), a collapsed far view, a rotated one"""
    from test_gpu_view_rd_sweep import cameras
    return [(I3, np.array([20.0, 0.0, 0.0])), (MIRROR, T0), (I3, np.array([0.0, 0.0, 3e7])), cameras(30.0)[2]]


@pytest.mark.gpu
def test_gpu_render_view_batch_adversarial_frames(dmc, port, exact):
    from oracle.oracle_py import synth_disp
    from test_gpu_render_view_batch import check
    H, W = 47, 61
    rs = np.random.RandomState(4)
    natural = port.filter_disp8u_depth32f(synth_disp(H, W, 2), 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0)
    odd = natural.copy()
    sel = rs.rand(H, W)
    odd[sel < 0.1] = np.nan; odd[(sel >= 0.1) & (sel < 0.15)] = np.inf; odd[(sel >= 0.15) & (sel < 0.2)] = -np.inf
    odd[(sel >= 0.2) & (sel < 0.3)] *= -1; odd[(sel >= 0.3) & (sel < 0.35)] = 0
    near = np.full((H, W), 1.0, F32)
    depth = np.stack([natural, odd, near, natural * 2])
    tex = colours(4 * H, W, 6).reshape(4, H, W, 3)
    for sub in (False, True):
        check(dmc, port, depth, tex, 80.0, batch_cameras(), sub, exact)
    d16 = np.stack([(natural * 10).astype(np.int16), (-natural * 10).astype(np.int16), rs.randint(-3000, 3000, (H, W)).astype(np.int16)])
    check(dmc, port, d16, tex[:3], 80.0, batch_cameras(), True, exact)


@pytest.mark.gpu
def test_gpu_render_view_batch_unsettled_frames(dmc, port, exact):
    """Chains longer than the sweep cap at frames 1 and 3 of a batch whose other frames settle: the batch reaches the
    serial finish, which must replay exactly the frames that did not settle."""
    from test_gpu_render_view_batch import port_view
    depth, chains = view_chain_batch()
    n, H, W = depth.shape
    tex = colours(n * H, W, 8).reshape(n, H, W, 3)
    K, R, t = view_intrinsics(H, W), I3[None], np.array([[VIEW_TX, 0.0, 0.0]])
    ctx = dmc.default_context()
    view_launches = 2 + base_launches(H, W)                  # reprojectXYZ, the render, fillSmallHole
    n0 = ctx.kernel_launches
    batch = dmc.renderViewBatch(depth, tex, VIEW_F, R, t, K, isSub=True, exact_divide=exact)
    assert ctx.kernel_launches - n0 == view_launches + sweep_cap(H, W) + 1          # the finish ran
    for i in range(n):
        n0 = ctx.kernel_launches
        alone = dmc.renderViewBatch(depth[i:i + 1], tex[i:i + 1], VIEW_F, R, t, K, isSub=True, exact_divide=exact)
        launches = ctx.kernel_launches - n0
        if i in chains:
            assert launches == view_launches + sweep_cap(H, W) + 1, (i, launches)
        else:
            assert launches < view_launches + sweep_cap(H, W), (i, launches)        # natural frames settle
        assert np.array_equal(batch[0, i], alone[0, 0]), (i, exact)
        assert np.array_equal(batch[0, i], port_view(port, depth[i], tex[i], VIEW_F, I3, t[0], K, True, not exact)), (i, exact)


@pytest.mark.gpu
def test_gpu_view_sweep_adversarial_frames(dmc, port):
    from oracle.oracle_py import synth_disp
    from test_gpu_view_rd_sweep import expect, intrinsics, params, texture_of
    H, W = 40, 56
    rs = np.random.RandomState(12)
    holes = synth_disp(H, W, 3); holes[rs.rand(H, W) < 0.3] = 0           # disparity 0: infinite depth
    disp = np.stack([synth_disp(H, W, 1), holes, np.full((H, W), 255, np.uint8), synth_disp(H, W, 2)])
    tex = np.stack([texture_of(d) for d in disp])
    f, cams, qs = 60.0, batch_cameras(), (20, 80)
    K = intrinsics(f, H, W)
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    batch = dmc.jpegViewRateDistortion(disp, tex, qs, params(dmc), f, R, t, K, isSub=True, exact_divide=True)
    for i in range(len(disp)):
        one = dmc.jpegViewRateDistortion(disp[i:i + 1], tex[i:i + 1], qs, params(dmc), f, R, t, K, isSub=True, exact_divide=True)
        for key in one:
            assert np.array_equal(batch[key][..., i:i + 1], one[key]), (i, key)
    nb, sc, sf = expect(port, disp, tex, qs, f, cams, K, True, False)
    assert np.array_equal(batch["bytes"], nb[0])
    assert np.array_equal(batch["sse_view_coded"], sc) and np.array_equal(batch["sse_view_filtered"], sf)
