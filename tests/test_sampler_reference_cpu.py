"""No-GPU checks of the float64 sampler reference (tests/_sampler_ref.py) that the GPU sampler tests compare the
kernels with, and of the samplers' host-side temperature check."""
import ctypes

import numpy as np
import pytest
from scipy import stats

from _sampler_ref import (RNG_POLICY, gumbel64, gumbel_max_ref, philox4x32_10, policy_words, uniform64,
                          uniform_valid_ref)


@pytest.mark.parametrize("counter,key,expected", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_matches_the_random123_known_answers(counter, key, expected):
    out = philox4x32_10(*[np.array([c], dtype=np.uint32) for c in counter], *key)
    assert tuple(int(w[0]) for w in out) == expected


def test_policy_counter_layout():
    """gid splits into (lo, hi), the third word is RNG_POLICY ^ step and the entry is the fourth"""
    gid, entry, seed, step = 2 ** 32 + 7, 123, 0x1234_5678_9ABC_DEF0, 0xFFFF_FFF0
    expect = philox4x32_10(np.array([7]), np.array([1]), np.array([RNG_POLICY ^ step]), np.array([entry]),
                           0x9ABC_DEF0, 0x1234_5678)[0]
    assert policy_words(np.array([gid]), np.array([entry]), seed, step)[0] == expect[0]


def test_uniform_extremes_are_exact_and_strictly_inside_the_unit_interval():
    words = np.array([0, 511, 512, 0xFFFFFE00, 0xFFFFFFFF], dtype=np.uint32)
    u = uniform64(words)
    assert u[0] == u[1] == 0.5 / 2 ** 23
    assert u[2] == 1.5 / 2 ** 23
    assert u[3] == u[4] == 1.0 - 0.5 / 2 ** 23
    assert (u.astype(np.float32).astype(np.float64) == u).all()  # exact in float32 as well
    g = gumbel64(words)
    assert np.isfinite(g).all()
    assert g[0] == pytest.approx(-np.log(-np.log(0.5 / 2 ** 23)), abs=0)
    assert 16.6 < g[-1] < 16.7 and -2.82 < g[0] < -2.80


def test_gumbel_reference_follows_the_standard_gumbel_quantiles():
    q = np.array([1e-6, 1e-3, 0.1, 0.5, 0.9, 0.999, 1 - 2 ** -20])
    k = np.floor(q * 2 ** 23).astype(np.uint32)  # u = (k + 0.5) / 2^23 is within 2^-24 of q
    g = gumbel64(k << np.uint32(9))
    u = uniform64(k << np.uint32(9))
    assert np.allclose(g, stats.gumbel_r.ppf(u), rtol=0, atol=1e-12)
    # a million consecutive counters: Kolmogorov-Smirnov against the standard Gumbel distribution
    words = policy_words(np.arange(1_000_000, dtype=np.uint64), np.zeros(1, dtype=np.uint64), 3, 1)
    assert stats.kstest(gumbel64(words), stats.gumbel_r.cdf).pvalue > 1e-3


def test_gumbel_max_ref_ties_empty_rows_and_minus_inf():
    n = 6
    logits = np.zeros((5, n))
    mask = np.zeros((5, n), dtype=np.uint8)
    mask[1, 4] = 1                            # one valid entry
    mask[2] = 1
    logits[2] = -np.inf                       # every valid logit -inf: the lowest valid index, NaN log-probability
    mask[3, [1, 3, 5]] = 1
    logits[3, [1, 3]] = -np.inf               # one finite entry wins
    mask[4, [1, 2]] = 1
    logits[4] = [np.nan, 5, 7, np.nan, 1, 2]  # invalid entries are never read
    with np.errstate(invalid="ignore"):
        ref = gumbel_max_ref(logits, mask, 1.0, np.arange(5), seed=1, step=2)
    assert ref.action.tolist()[:4] == [-1, 4, 0, 5]
    assert ref.gap[1] == np.inf and ref.gap[2] == np.inf and ref.gap[3] == np.inf
    assert ref.lse[0] == -np.inf and ref.lse[1] == 0.0 and ref.lse[2] == -np.inf
    assert ref.lse[3] == 0.0
    assert ref.lse[4] == pytest.approx(np.logaddexp(5, 7), abs=1e-15)
    # the draw itself: argmax of z + G with the entries' own words
    g = gumbel64(policy_words(np.uint64(4), np.array([1, 2], dtype=np.uint64), 1, 2))
    assert ref.action[4] == [1, 2][int(np.argmax(np.array([5.0, 7.0]) + g))]
    assert ref.gap[4] == pytest.approx(abs((5 + g[0]) - (7 + g[1])), abs=1e-12)

    # exact ties go to the lowest index: two entries with the same word cannot occur, so tie through the logits
    logits = np.array([[0.0, 0.0]])
    mask = np.ones((1, 2), dtype=np.uint8)
    g = gumbel64(policy_words(np.uint64(0), np.array([0, 1], dtype=np.uint64), 0, 0))
    logits[0, 1] = g[0] - g[1]  # z1 + G1 == z0 + G0 in float64
    ref = gumbel_max_ref(logits, mask, 1.0, [0], seed=0, step=0)
    assert ref.action[0] == 0 and ref.gap[0] == pytest.approx(0.0, abs=1e-15)


def test_gumbel_max_ref_temperature_scales_z_only():
    rng = np.random.default_rng(0)
    logits = rng.standard_normal((64, 40))
    mask = (rng.random((64, 40)) < 0.5).astype(np.uint8)
    a = gumbel_max_ref(logits, mask, 0.5, np.arange(64), 9, 9)
    b = gumbel_max_ref(logits * 2.0, mask, 1.0, np.arange(64), 9, 9)
    assert np.array_equal(a.action, b.action) and np.allclose(a.lse, b.lse, rtol=0, atol=1e-12)


def test_uniform_valid_ref_conventions():
    mask = np.zeros((4, 33), dtype=np.uint8)
    mask[1, 32] = 1
    mask[2, [0, 5, 31, 32]] = 1
    mask[3] = 1
    words = np.array([0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0], dtype=np.uint32)
    assert uniform_valid_ref(mask, words).tolist() == [-1, 32, 32, 0]
    assert uniform_valid_ref(mask, words, empty=35)[0] == 35
    words = np.array([0, 0, 0x40000000, 0x80000000], dtype=np.uint32)  # t = 1 of 4 and t = 16 of 33
    assert uniform_valid_ref(mask, words).tolist() == [-1, 32, 5, 16]


@pytest.mark.parametrize("temperature", [0.0, -1.0, float("nan"), 1e-40, 2.0 ** -128])
def test_samplers_reject_temperatures_without_a_finite_reciprocal(temperature):
    """z = logit * (1 / T): a subnormal T would turn every 0-valued logit into NaN.  The checks run before any launch,
    so dummy non-null pointers and zero games reach them without a device."""
    from stratego_env_b200 import _lib
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)
    assert lib.sx_sample_logits(dummy, 0, dummy, 0, 8, 0, 0, 0, temperature, dummy, None, None) != 0
    assert b"temperature" in lib.sx_last_error()
    st = _lib.SxState(16, 16, 16)
    assert lib.sx_sample_policy(dummy, st, 0, 0, dummy, 0, 0, 0, temperature, dummy, None, None) != 0
    assert b"temperature" in lib.sx_last_error()
    # a normal temperature passes the check (zero games: nothing is launched)
    assert lib.sx_sample_logits(dummy, 0, dummy, 0, 8, 0, 0, 0, 1e-30, dummy, None, None) == 0
    assert lib.sx_sample_policy(dummy, st, 0, 0, dummy, 0, 0, 0, 1e-30, dummy, None, None) == 0
