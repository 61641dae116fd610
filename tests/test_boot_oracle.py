"""The NumPy restatement of the bootstrap (tests/boot_oracle.py) on its own: SplitMix64 against its published values,
the balance of the Rademacher signs, and the summary against hand-worked cases."""
import numpy as np
import pytest

import boot_oracle as O


def test_splitmix64_published_values():
    h = O.splitmix64(0, np.arange(3, dtype=np.uint64))
    assert [int(x) for x in h] == [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F]


def test_signs_are_balanced_per_echo():
    """10^5 words: every one of the 64 bits is set in half of them to within 5 standard deviations (sd = 158)."""
    s = O.signs(1000, 100, 64, seed=12345, voxel_offset=7).reshape(-1, 64)
    assert s.shape == (100000, 64)
    ones = s.sum(axis=0)
    assert np.all(np.abs(ones - 50000) < 5 * np.sqrt(100000 * 0.25)), ones


def test_replicates_keyed_on_the_global_voxel_position():
    rng = np.random.default_rng(1)
    sig = rng.uniform(50, 100, (6, 32))
    est = sig + rng.normal(0, 1, sig.shape)
    fa = np.arange(6, dtype=np.int32)
    whole, whole_fa = O.resample(sig, est, fa, 5, seed=3)
    a, _ = O.resample(sig[:2], est[:2], fa[:2], 5, seed=3)
    b, b_fa = O.resample(sig[2:], est[2:], fa[2:], 5, seed=3, voxel_offset=2)
    assert np.array_equal(np.concatenate([a, b]), whole) and np.array_equal(b_fa, whole_fa[10:])
    assert not np.array_equal(O.resample(sig, est, fa, 5, seed=4)[0], whole)
    # each echo is est + r or est - r
    r = (sig - est)[:, None, :]
    w = whole.reshape(6, 5, 32)
    assert np.all((w == est[:, None, :] + r) | (w == est[:, None, :] - r))


def _one(x):
    return O.summarise_values(np.asarray(x, dtype=np.float64))


def test_summary_hand_cases():
    assert _one([]) == (0.0, 0.0, 0.0, 0.0)
    assert _one([3.5]) == (3.5, 0.0, 3.5, 3.5)
    m, s, lo, hi = _one([1.0, 3.0])
    # idx = 0.025 and 0.975: gamma < 0.5 -> a + (b - a) g; gamma >= 0.5 -> b - (b - a)(1 - g)
    assert (m, s) == (2.0, np.sqrt(2.0)) and lo == 1.0 + 2.0 * 0.025 and hi == 3.0 - 2.0 * (1.0 - 0.975)
    # odd n, unsorted input, ties
    x = [4.0, 1.0, 4.0, 2.0, 4.0]
    m, s, lo, hi = _one(x)
    assert m == 3.0 and s == np.sqrt(((1.0 ** 2) * 3 + 4.0 + 1.0) / 4)
    assert lo == np.percentile(x, 2.5) and hi == 4.0
    # even n
    x = [0.1 * k for k in range(10)][::-1]
    assert _one(x)[2:] == tuple(np.percentile(x, [2.5, 97.5]))
    # gamma exactly 0.5: n = 21 -> idx = 20 * 0.025 = 0.5; the b - (b - a)(1 - g) branch
    x = np.arange(21.0) * 3.0 + 1.0
    idx = 20 * (2.5 / 100)
    assert idx == 0.5
    assert _one(x)[2] == 4.0 - (4.0 - 1.0) * (1 - 0.5)
    # NaN among the values: all four NaN
    assert all(np.isnan(_one([1.0, np.nan, 2.0])))


def test_summary_skips_skipped_replicates():
    B = 4
    maps = np.arange(2 * B * 6, dtype=np.float64).reshape(2 * B, 6)
    status = np.array([0, 1, 4, 1 | 2, 1, 1, 1, 1], dtype=np.uint32)   # ITMAX alone is valid; SKIPPED is not
    stats, n = O.summary(maps, status, B)
    assert list(n) == [2, 0]
    assert np.array_equal(stats[1], np.zeros((6, 4)))
    for m in range(6):
        assert tuple(stats[0, m]) == _one(maps[[0, 2], m])


@pytest.mark.parametrize("n", [2, 3, 40, 41, 100, 1024])
def test_summary_matches_numpy_statistics(n):
    x = np.random.default_rng(n).normal(0.2, 0.05, n)
    m, s, lo, hi = _one(x)
    assert abs(m - np.mean(x)) < 1e-15 and abs(s - np.std(x, ddof=1)) < 1e-15
    assert (lo, hi) == tuple(np.percentile(x, [2.5, 97.5]))
