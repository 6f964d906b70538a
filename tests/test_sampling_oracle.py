"""The float64 restatement of the device samplers (oracle/ppo_ref.py): vectorised Philox4x32-10, the counter layout,
Box-Muller and the categorical inverse CDF, on the CPU.  tests/test_sampling_gpu.py checks the kernels against it."""
import numpy as np
import pytest
from scipy import stats

from oracle import ppo_ref as R

# (seed, gid, step, word, value of word >> 8): counters whose sampler block hits the ends of the 24-bit uniforms.
# Word 0 is the categorical u and Box-Muller's first radius, word 1 the first angle, word 2 the second radius.
# Found with the vectorised Philox, a few seconds per 2^24 counters:
#   h = R.sampler_words_np(77, np.arange(1 << 24, dtype=np.uint64), step) >> 8
#   np.nonzero(h[0] == 0), np.nonzero(h[0] >= 0xFFFFF0), np.nonzero(h[1] == 0), np.nonzero(h[2] == 0)
# for step = 5 .. 12.
EXTREME_COUNTERS = [
    (77, 16475180, 6, 0, 0x000000),      # u = 0
    (77, 968600, 7, 0, 0x000000),
    (77, 3475739, 6, 0, 0xFFFFFF),       # u = 1 - 2^-24, the largest
    (77, 14825738, 9, 0, 0xFFFFFF),
    (77, 7816114, 12, 0, 0xFFFFFF),
    (77, 15013369, 5, 0, 0xFFFFFC),
    (77, 11861222, 5, 0, 0xFFFFF9),
    (77, 8058961, 5, 1, 0x000000),       # angle 2 pi 2^-25
    (77, 13409660, 5, 2, 0x000000),      # smallest second radius argument
]
Z_MAX = float(np.sqrt(-2.0 * np.log(2.0 ** -25)))     # |z| bound of Box-Muller on u in [2^-25, 1 - 2^-25]


def test_vectorised_philox_equals_scalar():
    rng = np.random.default_rng(0)
    c = rng.integers(0, 2 ** 32, (4, 2000), dtype=np.uint64)
    k = rng.integers(0, 2 ** 32, (2, 2000), dtype=np.uint64)
    c[:, :3], k[:, :3] = 0xFFFFFFFF, 0xFFFFFFFF
    c[:, 3:6], k[:, 3:6] = 0, 0
    got = R.philox4x32_10_np(*c, *k)
    assert got.dtype == np.uint32 and got.shape == (4, 2000)
    for i in range(2000):
        assert tuple(int(w) for w in got[:, i]) == R.philox4x32_10(c[:, i], k[:, i]), i
    # known answers (Salmon et al., SC'11 / Random123 kat_vectors), as tests/test_oracle_ppo.py checks the scalar form
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        assert tuple(int(w) for w in R.philox4x32_10_np(*ctr, *key)) == want


@pytest.mark.parametrize("seed", [77, 2 ** 40 + 5, 2 ** 64 - 1])
def test_counter_layout_of_the_samplers(seed):
    ids = np.array([0, 1, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 17, 2 ** 63 + 3, 2 ** 64 - 1], dtype=np.uint64)
    steps = np.array([0, 5, 2 ** 32 + 1, 2 ** 33, 2 ** 40 + 9, 7, 2 ** 64 - 1], dtype=np.uint64)
    w = R.sampler_words_np(seed, ids, steps)
    for i in range(len(ids)):
        assert tuple(int(x) for x in w[:, i]) == R.sampler_words(seed, int(ids[i]), int(steps[i]))
    for blk in (1, 3):
        c = R.sampler_counter(ids, steps, blk)
        assert np.array_equal(c[3], (steps >> np.uint64(32)) ^ np.uint64(blk << 24))
        assert np.array_equal(c[0], ids & np.uint64(0xFFFFFFFF)) and np.array_equal(c[1], ids >> np.uint64(32))
        wb = R.sampler_words_np(seed, ids, steps, blk)
        for i in range(len(ids)):
            want = R.philox4x32_10((int(c[0][i]), int(c[1][i]), int(c[2][i]), int(c[3][i])), (seed & 0xFFFFFFFF, seed >> 32))
            assert tuple(int(x) for x in wb[:, i]) == want
        assert (wb != w).all()


@pytest.mark.parametrize("seed,gid,step,word,value", EXTREME_COUNTERS)
def test_extreme_counters(seed, gid, step, word, value):
    w = R.sampler_words(seed, gid, step)
    assert w[word] >> 8 == value
    assert tuple(int(x) for x in R.sampler_words_np(seed, gid, step)) == w
    z = R.normal4_f64(np.array(w, dtype=np.uint32))
    assert np.isfinite(z).all() and (np.abs(z) <= Z_MAX).all(), z
    r01, r23 = np.hypot(z[0], z[1]), np.hypot(z[2], z[3])
    if word == 0 and value == 0:
        assert r01 == pytest.approx(Z_MAX, rel=1e-15)
        assert float(R.u01(w[0])) == 0.0
    if word == 0 and value == 0xFFFFFF:
        assert r01 == pytest.approx(2.0 ** -12, rel=1e-6)            # sqrt(-2 ln(1 - 2^-25))
        assert float(R.u01(w[0])) == 1 - 2.0 ** -24
    if word == 1:                                                   # angle 2 pi 2^-25: z1 / z0 = tan(2 pi 2^-25)
        assert z[1] / z[0] == pytest.approx(2 * np.pi * 2.0 ** -25, rel=1e-12)
    if word == 2:
        assert r23 == pytest.approx(Z_MAX, rel=1e-15)


def test_box_muller_restatement_is_standard_normal():
    w = R.sampler_words_np(3, np.arange(1 << 18, dtype=np.uint64), 11)
    z = R.normal4_f64(w)
    assert z.shape == (1 << 18, 4)
    for d in range(4):
        assert stats.kstest(z[:, d], "norm").pvalue > 1e-3, d
    c = np.corrcoef(z.T)
    assert np.abs(c - np.eye(4)).max() < 5 / np.sqrt(len(z))
    # hand-computed words: u1 = u2 = 1/2 -> z = (-sqrt(2 ln 2), 0)
    half = np.uint32(0x80 << 24)
    z = R.normal4_f64(np.array([half - 128, half - 128, half - 128, half - 128], dtype=np.uint32))
    ang = 2 * np.pi * 0.5 * (1 - 2.0 ** -24)
    r = np.sqrt(-2 * np.log(0.5 * (1 - 2.0 ** -24)))
    np.testing.assert_allclose(z, [r * np.cos(ang), r * np.sin(ang)] * 2, rtol=1e-15)


def test_categorical_inverse_cdf():
    p = np.array([[0.2, 0.3, 0.5]] * 7 + [[0.0, 0.25, 0.75]] * 2 + [[0.5, 0.5 - 2.0 ** -30, 0.0]] * 2)
    u = np.array([0.0, 0.1, 0.2, 0.2 + 1e-12, 0.5, 0.75, 1 - 2.0 ** -24, 0.0, 0.25, 0.75, 1 - 2.0 ** -24])
    cls, margin = R.categorical_icdf(p, u)
    # first k with u < P_0 + .. + P_k; a dead first class is never taken at u = 0, a draw past the total takes class 1 of
    # [0.5, 0.5 - 2^-30, 0], not the dead class 2
    assert cls.tolist() == [0, 0, 1, 1, 2, 2, 2, 1, 2, 1, 1]
    np.testing.assert_allclose(margin[:7], [0.2, 0.1, 0.0, 1e-12, 0.0, 0.25, 0.5 - 2.0 ** -24], atol=1e-15)
    assert margin[7] == 0.0 and margin[8] == 0.0
    cls, margin = R.categorical_icdf(np.ones((3, 1)), np.array([0.0, 0.5, 1 - 2.0 ** -24]))
    assert cls.tolist() == [0, 0, 0] and np.isinf(margin).all()
    # frequencies of the restated rule over restated uniforms follow the probabilities
    pr = np.array([0.1, 0.2, 0.3, 0.4])
    w = R.sampler_words_np(5, np.arange(1 << 18, dtype=np.uint64), 0)
    uu = (w[0] >> 8).astype(np.float64) * 2.0 ** -24
    cls, _ = R.categorical_icdf(np.broadcast_to(pr, (len(uu), 4)), uu)
    assert stats.chisquare(np.bincount(cls, minlength=4), pr * len(uu)).pvalue > 1e-3
