"""The numpy Philox restatement (oracle/philox.py) against the Random123 known answers, and the ranges of the
policy and env draws built on it.  CPU only: the GPU tests compare the library's device draws with these."""
import numpy as np
import pytest

from oracle import philox as P

# Random123 kat_vectors, philox4x32_10: counter, key, output
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(ctr, key, want):
    got = P.philox4x32_10(*ctr, *key)
    assert [int(x) for x in got] == list(want)
    assert all(x.dtype == np.uint32 for x in got)


def test_philox_vectorised_equals_scalar():
    """Arrays of counters give, element by element, what one counter at a time gives (no lane mixes with another)."""
    rng = np.random.default_rng(0)
    c = rng.integers(0, 2**32, (4, 37), dtype=np.uint64)
    k = rng.integers(0, 2**32, 2, dtype=np.uint64)
    vec = P.philox4x32_10(*c, *k)
    for i in range(37):
        one = P.philox4x32_10(*(int(x[i]) for x in c), int(k[0]), int(k[1]))
        assert [int(v[i]) for v in vec] == [int(x) for x in one]


def test_u53_range_and_resolution():
    # extremes: 0 and the largest double below 1
    assert P.u53(0, 0) == 0.0
    top = P.u53(0xFFFFFFFF, 0xFFFFFFFF)
    assert top < 1.0 and top == 1.0 - 2.0**-53
    # the lowest used bit of each word moves u by exactly one step of 2^-53 resp. 2^-26
    assert P.u53(0, 1 << 6) == 2.0**-53 and P.u53(0, (1 << 6) - 1) == 0.0
    assert P.u53(1 << 5, 0) == 2.0**-27 and P.u53((1 << 5) - 1, 0) == 0.0


@pytest.mark.parametrize("n_act", [1, 3, 4, 7, 8])
def test_policy_draws_ranges(n_act):
    ra, u = P.policy_draws(200_000, n_act, seed=3, step=9)
    assert ra.min() >= 0 and ra.max() < n_act and (n_act == 1 or ra.max() == n_act - 1)
    assert u.min() >= 0.0 and u.max() < 1.0
    # 53 bits: every u is a whole multiple of 2^-53, and the low bits are in use
    m = u * 2.0**53
    assert np.array_equal(m, np.floor(m))
    assert (m.astype(np.uint64) & np.uint64(1)).mean() > 0.45
    assert np.abs(np.bincount(ra, minlength=n_act) / ra.size - 1.0 / n_act).max() < 0.01
    assert abs(u.mean() - 0.5) < 0.01


def test_policy_draws_counter_words():
    """u does not depend on n_act; the row index feeds words 0/1, the step words 2/3 (the high words count)."""
    rows = np.array([0, 5, 2**32 + 5], dtype=np.uint64)
    ra4, u4 = P.policy_draws(rows, 4, seed=2**40 + 7, step=2**32 + 5)
    ra7, u7 = P.policy_draws(rows, 7, seed=2**40 + 7, step=2**32 + 5)
    assert np.array_equal(u4, u7)
    _, ulo = P.policy_draws(rows, 4, seed=2**40 + 7, step=5)
    _, uhi = P.policy_draws(rows, 4, seed=7, step=2**32 + 5)
    assert not np.any(ulo == u4) and not np.any(uhi == u4)
    assert u4[1] != u4[2]  # the row's high word counts
    r0, r1, r2, _ = P.philox4x32_10(5, 1, 5, 1 ^ 0x5BD1E995, 0xDEADBEEF ^ 7, 0xA5A5A5A5 ^ (2**40 >> 32))
    assert u4[2] == P.u53(r1, r2) and ra4[2] == (int(r0) * 4) >> 32


def test_env_draws_layout_and_ranges():
    B, A, N = 9, 45, 20
    s, t, z = P.env_draws(B, A, N, seed=11, step=3)
    assert s.shape == t.shape == z.shape == (B, A) and s.dtype == np.int32 and z.dtype == np.float64
    assert s.min() >= 0 and s.max() < N and t.min() >= 0 and t.max() < N
    assert z.min() >= 0 and z.max() < 1
    r0, r1, r2, r3 = P.philox4x32_10(7, 4, 3, 0, 11, 0)  # slot 7 of env 4
    assert s[4, 7] == (int(r0) * N) >> 32 and t[4, 7] == (int(r1) * N) >> 32 and z[4, 7] == P.u53(r2, r3)
    # the step's high word is counter word 3
    _, _, zh = P.env_draws(B, A, N, seed=11, step=2**32 + 3)
    assert not np.any(zh == z)
    # a larger batch starts with the same envs
    s2, t2, z2 = P.env_draws(2 * B, A, N, seed=11, step=3)
    assert np.array_equal(s2[:B], s) and np.array_equal(t2[:B], t) and np.array_equal(z2[:B], z)
