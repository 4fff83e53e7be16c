"""The tile order of the one-launch products emit (k_multi_order in magot_b200/csrc/mg_emit.cu), restated in numpy int64 and
checked without a GPU.  Tile t of job j (n_j tiles, lag_j) has the key floor((2t + 1) * 2^30 / (2 n_j)) + lag_j; the kernel
gives it the rank t + (tiles of earlier jobs with key <= K) + (tiles of later jobs with key < K), from closed-form counts and
no sort.  If that ever dropped or doubled a rank, a tile of some text would never be written."""
import bisect

import numpy as np
import pytest

SH = 30                                               # MULTI_SH
NMAX = 1 << 28                                        # tiles of one launch: order words are job << 28 | tile


def lags_of(ppm, present):
    """m.lag of mg_emit_products_device: job 1 behind job 0 when job 0 runs, job 2 behind job 1 when job 1 runs."""
    lag = (ppm << SH) // 1000000
    l1 = lag if present[0] else 0
    return [0, l1, l1 + (lag if present[1] else 0)]


def keys(n, lag):
    t = np.arange(n, dtype=np.int64)
    return (((2 * t + 1) << SH) // (2 * n)) + lag


def count_lt(K, n, lag):
    """multi_count_lt: tiles of a job whose key is < K (K an int64 array)."""
    Kp = np.asarray(K, dtype=np.int64) - lag
    if n == 0:
        return np.zeros_like(Kp)
    q = (Kp * (2 * n) - 1) >> SH
    return np.where(Kp <= 0, 0, np.minimum(n, (q + 1) >> 1))


def ranks(ns, lags):
    """rank of every tile, job by job, as k_multi_order computes it."""
    out = []
    for j in range(3):
        if ns[j] == 0:
            out.append(np.zeros(0, dtype=np.int64))
            continue
        K = keys(ns[j], lags[j])
        r = np.arange(ns[j], dtype=np.int64)
        for jj in range(3):
            if jj != j:
                r = r + count_lt(K + 1 if jj < j else K, ns[jj], lags[jj])
        out.append(r)
    return out


def check_order(ns, lags):
    rs = ranks(ns, lags)
    N = sum(ns)
    allr = np.concatenate(rs)
    # a bijection onto [0, N): every rank taken exactly once
    assert allr.size == N
    if N:
        assert allr.min() == 0 and allr.max() == N - 1
        assert np.bincount(allr, minlength=N).max() == 1
    # consistent with the key order, ties by (job, tile)
    K = np.concatenate([keys(ns[j], lags[j]) for j in range(3) if ns[j]] or [np.zeros(0, np.int64)])
    J = np.concatenate([np.full(ns[j], j, dtype=np.int64) for j in range(3)])
    T = np.concatenate([np.arange(ns[j], dtype=np.int64) for j in range(3)])
    order = np.lexsort((T, J, K))
    assert np.array_equal(allr[order], np.arange(N, dtype=np.int64))


PPMS = [0, 1, 1_000_000]


@pytest.mark.parametrize("ppm", PPMS)
def test_multi_order_permutation(ppm):
    rng = np.random.default_rng(20 + ppm % 97)
    cases = [(1, 1, 1), (1, 0, 0), (0, 1, 0), (0, 0, 1), (0, 0, 0), (7, 3, 2), (1, 1000, 1), (1000, 1, 333), (2, 2, 2),
             (1 << 20, 1, 0), (0, 1 << 20, 3), (12345, 0, 6789)]
    for _ in range(6):                                 # random sizes up to ~2^22 tiles in all, some jobs empty
        ns = [int(x) for x in rng.integers(0, 1 << 21, size=3)]
        ns[int(rng.integers(0, 4)) % 3] *= int(rng.integers(0, 2))
        cases.append(tuple(ns))
    for _ in range(40):                                # many small ones: ties are dense
        cases.append(tuple(int(x) for x in rng.integers(0, 40, size=3)))
    for ns in cases:
        for present in ((ns[0] > 0, ns[1] > 0), (True, True), (False, True), (True, False)):
            # a job can be present (its plan's size on the host is a capacity > 0) with no tile on the device
            check_order(list(ns), lags_of(ppm, present))


def _key_exact(t, n, lag):
    return ((2 * t + 1) << SH) // (2 * n) + lag


def _count_lt_exact(K, n, lag):
    """independent of the closed form: keys grow with t, so bisect them (Python integers, no overflow)."""
    if n == 0:
        return 0

    class Keys(object):
        def __len__(self):
            return n

        def __getitem__(self, t):
            return _key_exact(t, n, lag)
    return bisect.bisect_left(Keys(), K)


@pytest.mark.parametrize("ppm", PPMS)
def test_multi_order_large_counts_no_overflow(ppm):
    """Single ranks at up to 2^28 tiles: the int64 closed form against exact integer arithmetic.  At 1 000 000 ppm job 2 lags by
    2^31, so K * 2n reaches ~3 * 2^59."""
    shapes = [(NMAX - 3, 1, 1), (1, NMAX - 3, 1), (1, 1, NMAX - 3), (NMAX // 3, NMAX // 3, NMAX // 3 - 1),
              (NMAX // 2, 0, NMAX // 2 - 1), (0, NMAX - 1, 0), (5, 7, NMAX - 13)]
    for ns in shapes:
        present = (ns[0] > 0, ns[1] > 0)
        lags = lags_of(ppm, present)
        for j in range(3):
            n = ns[j]
            if n == 0:
                continue
            for t in sorted(t for t in {0, 1, n // 3, n // 2, n - 2, n - 1} if 0 <= t < n):
                K = _key_exact(t, n, lags[j])
                assert int(keys(n, lags[j])[t] if n < (1 << 16) else
                           ((((2 * np.int64(t) + 1) << SH) // (2 * np.int64(n))) + lags[j])) == K
                want = t + sum(_count_lt_exact(K + 1 if jj < j else K, ns[jj], lags[jj]) for jj in range(3) if jj != j)
                got = t + sum(int(count_lt(np.array([K + 1 if jj < j else K]), ns[jj], lags[jj])[0]) for jj in range(3) if jj != j)
                assert got == want, (ns, j, t)
                assert 0 <= got < sum(ns)
