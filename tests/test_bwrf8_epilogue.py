"""CPU proof of the two integer divisions of the 8-bit range filter (dmc_bwrf8u_h2.cu), against the reference's
RNE(float(sum) / float(N)) (_mm_div_ps, then _mm_cvtps_epi32), for every pair the filter can reach at radius 1..10 and
any threshold: N = 1 .. 317 accepted taps (317 = the taps of the radius-10 disc), sum = 0 .. 255 * N.

  rne_div   the tap loop's epilogue: t = 15 * sum, n = 15 * N (the counter counts 15 per tap), q = RNE(t * r) with r any
            float within one ulp of 1/n (rcp.approx.f32), e = t - q * n, then q +- 1 toward the nearest, ties to even.
  flat      the flat-warp path: N = ntaps (odd), out = (sum + ntaps // 2) // ntaps in integers."""
import numpy as np

NMAX = 317


def ntaps(r):
    n = 0
    for dy in range(-r, r + 1):
        lim, j = r * r - dy * dy, 0
        while (j + 1) * (j + 1) <= lim:
            j += 1
        n += 2 * j + 1
    return n


def reference(s, n):
    return np.rint(s.astype(np.float32) / np.float32(n)).astype(np.int64)


def rne_div(t, n, r):
    """the kernel's rne_div in exact arithmetic: the FFMA t * r + 1.5 * 2^23 rounds once, to an integer (t * r is exact
    in double: 24 x 24 significant bits); the FFMA t - q * n is exact (integers below 2^24)"""
    q = np.rint(t * np.float64(r))
    e = t - q * n
    hn = 0.5 * n
    odd = np.mod(q, 2) == 1
    return (q + ((e > hn) | ((e == hn) & odd)) - ((e < -hn) | ((e == -hn) & odd))).astype(np.int64)


def test_ntaps():
    assert [ntaps(r) for r in range(1, 11)][-1] == NMAX
    assert all(ntaps(r) % 2 == 1 for r in range(1, 11))
    # the flat path's 16-bit fields hold sum(v - m) <= ntaps * 2 * th with th <= 2048 // (2r + 1)
    assert all(ntaps(r) * 2 * (2048 // (2 * r + 1)) < 65536 for r in range(1, 11))


def test_rne_div_every_reachable_pair():
    for N in range(1, NMAX + 1):
        s = np.arange(0, 255 * N + 1, dtype=np.int64)
        want = reference(s, N)
        t, n = (15 * s).astype(np.float64), float(15 * N)
        r0 = np.float32(1.0) / np.float32(n)
        for r in (np.nextafter(r0, np.float32(0)), r0, np.nextafter(r0, np.float32(1))):
            got = rne_div(t, n, r)
            bad = np.flatnonzero(got != want)
            assert bad.size == 0, "N=%d r=%r: sum=%d gives %d, want %d" % (N, r, s[bad[0]], got[bad[0]], want[bad[0]])


def test_flat_path_division():
    for r in range(1, 11):
        N = ntaps(r)
        s = np.arange(0, 255 * N + 1, dtype=np.int64)
        assert np.array_equal((s + N // 2) // N, reference(s, N)), r
        # with the footprint minimum m taken out of every tap: m + (sum(v - m) + N // 2) // N
        for m in (0, 1, 77, 255):
            sm = s[s >= N * m] - N * m
            assert np.array_equal(m + (sm + N // 2) // N, reference(s[s >= N * m], N)), (r, m)
