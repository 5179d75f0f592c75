"""CPU: the NumPy reference of the fused actor's Gaussian draws (``oracle_np.philox_normal_pair``), which the GPU tests in
tests/test_random_streams_gpu.py compare the kernels with.  It reuses ``philox4x32``, which the Random123 known-answer
test in tests/test_oracle_golden.py pins; here its keying, its float32 rounding of the radius uniform, its distribution
and the tail targets the GPU tests run are checked."""
import math

import numpy as np
import scipy.stats

from oracle import oracle_np as o

SEED = 0xD1B54A32D192ED03          # both key words non-zero, above 2^63
R_MAX = math.sqrt(-2.0 * math.log(2.0 ** -25))   # the largest radius: k1 = 0, u1 = 2^-25

# Keys whose 24-bit words hit the tails of Box-Muller, found by tests/golden/gen_random_tail_targets.py: (word, k, env id,
# stream, blk) at seed TAIL_SEED, step TAIL_STEP.  k1 = 0xFFFFFF gives u1 = 1 (r = 0); k1 = 0xFFFFFE - 2 (j - 1) the eight
# u1 values 1 - j 2^-23 below it, where ln u1 is smaller than the documented error of __logf; k1 = 0, 1 the largest
# radii; k2 = 0, 2^22, 2^23, 3 2^22, 2^24 - 1 the angles 0, pi / 2, pi, 3 pi / 2 and just below 2 pi.
TAIL_SEED, TAIL_STEP = SEED, 0x80000005
TAIL_TARGETS = [
    ("k1", 0xFFFFFF, 0xFE1B43F3, 7, 2),
    ("k1", 0xFFFFFE, 0xFE526023, 8, 0),
    ("k1", 0xFFFFFC, 0xFE2F5742, 7, 1),
    ("k1", 0xFFFFFA, 0xFE25A279, 8, 0),
    ("k1", 0xFFFFF8, 0xFE494B41, 8, 1),
    ("k1", 0xFFFFF6, 0xFE836FFE, 8, 0),
    ("k1", 0xFFFFF4, 0xFE5BCB26, 8, 0),
    ("k1", 0xFFFFF2, 0xFE010111, 8, 2),
    ("k1", 0xFFFFF0, 0xFE029E9D, 8, 2),
    ("k1", 0x000000, 0xFE0D8516, 7, 2),
    ("k1", 0x000001, 0xFE48E75A, 7, 1),
    ("k2", 0x000000, 0xFE3C060B, 7, 0),
    ("k2", 0x400000, 0xFE0A7084, 7, 1),
    ("k2", 0x800000, 0xFE0F2C9A, 8, 1),
    ("k2", 0xC00000, 0xFE112AE7, 8, 3),
    ("k2", 0xFFFFFF, 0xFE17F3C4, 7, 0),
]


def test_radius_uniform_mirrors_the_float32_rounding():
    """u1 = (float(k1) + 0.5f) 2^-24 in float32: k1 = 2^24 - 1 rounds to u1 = 1 exactly, the upper half [0.5, 1] takes
    2^22 + 1 values (the add rounds to even for k1 >= 2^23), the lower half is exact and never reaches 0."""
    assert o.normal_pair_u1(2 ** 24 - 1) == np.float32(1.0)
    assert o.normal_pair_u1(2 ** 24 - 2) == o.normal_pair_u1(2 ** 24 - 3) == np.float32(1.0 - 2.0 ** -23)
    assert o.normal_pair_u1(0) == np.float32(2.0 ** -25)
    upper = o.normal_pair_u1(np.arange(2 ** 23, 2 ** 24))
    assert upper.dtype == np.float32 and upper.min() == 0.5 and upper.max() == 1.0
    assert np.unique(upper).size == 2 ** 22 + 1
    lower = np.arange(2 ** 23, dtype=np.float64)
    assert np.array_equal(o.normal_pair_u1(np.arange(2 ** 23)).astype(np.float64), (lower + 0.5) * 2.0 ** -24)


def test_normal_pair_keying_matches_philox_uniform():
    """Stream 0 of the pair reference draws the words philox_uniform draws (value 4 blk + 0 is k1, 4 blk + 1 is k2), at
    env ids on both sides of 2^32, steps above 2^31 and a seed with both words non-zero; the stream moves the counter."""
    env = np.concatenate([np.arange(2 ** 32 - 300, 2 ** 32 + 300), np.arange(2 ** 63 - 50, 2 ** 63 + 50)]).astype(np.uint64)
    for step in (0, 1, 2 ** 31 + 7, 2 ** 32 - 1):
        u = o.philox_uniform(SEED, env, np.full(env.shape, step, dtype=np.uint64), 16)
        for blk in range(4):
            k1, k2, z0, z1 = o.philox_normal_pair(SEED, env, step, blk, 0)
            assert np.array_equal(k1 * 2.0 ** -24, u[:, 4 * blk]) and np.array_equal(k2 * 2.0 ** -24, u[:, 4 * blk + 1])
            k1s, _, _, _ = o.philox_normal_pair(SEED, env, step, blk, 7)
            assert np.mean(k1s == k1) < 0.01
    # the high words of the seed and of the env id both take part
    k_full = o.philox_normal_pair(SEED, env, 5, 0, 7)[0]
    assert np.mean(o.philox_normal_pair(SEED & 0xFFFFFFFF, env, 5, 0, 7)[0] == k_full) < 0.01
    hi = env >= np.uint64(2 ** 32)
    assert np.mean(o.philox_normal_pair(SEED, env[hi] & np.uint64(0xFFFFFFFF), 5, 0, 7)[0] == k_full[hi]) < 0.01


def test_normal_pair_values_and_distribution():
    """z0 = r cos(theta), z1 = r sin(theta) from the words; 1e6 draws of each component pass a KS test against N(0, 1)
    and stay within the largest radius sqrt(-2 ln 2^-25) = 5.8870."""
    env = np.arange(2 ** 32 - 2 ** 17, 2 ** 32 + 2 ** 17, dtype=np.uint64)
    zs = []
    for blk in range(4):
        k1, k2, z0, z1 = o.philox_normal_pair(SEED, env, 3, blk, 7)
        r = np.sqrt(-2.0 * np.log((k1.astype(np.float64) + 0.5) * 2.0 ** -24))   # k1 + 0.5 is exact below 2^23
        th = 2.0 * np.pi * k2 * 2.0 ** -24
        low = k1 < 2 ** 23
        assert np.allclose(z0[low], (r * np.cos(th))[low], rtol=0, atol=1e-15)
        assert np.allclose(z1[low], (r * np.sin(th))[low], rtol=0, atol=1e-15)
        zs += [z0, z1]
    z = np.concatenate(zs)
    assert z.size > 2e6
    for comp in (z[0::2][:10 ** 6], z[1::2][:10 ** 6]):
        assert scipy.stats.kstest(comp, "norm").pvalue > 1e-3
    assert np.abs(z).max() <= R_MAX
    assert abs(R_MAX - 5.8870) < 1e-4


def test_tail_targets_produce_their_words():
    """Each committed tail target draws its claimed k in its claimed word; u1 = 1 gives the pair (0, 0), k1 = 0 the
    largest radius, and the quadrant-edge angles their exact axes."""
    assert len(TAIL_TARGETS) == 16
    for word, k, env, stream, blk in TAIL_TARGETS:
        k1, k2, z0, z1 = o.philox_normal_pair(TAIL_SEED, [env], TAIL_STEP, blk, stream)
        assert int((k1 if word == "k1" else k2)[0]) == k, (word, k, env)
        r = math.hypot(z0[0], z1[0])
        if word == "k1" and k == 0xFFFFFF:
            assert z0[0] == 0.0 and z1[0] == 0.0
        if word == "k1" and k == 0:
            assert abs(r - R_MAX) < 1e-12
        if word == "k2" and k % 2 ** 22 == 0:
            q = k // 2 ** 22      # theta = q pi / 2
            assert abs(z0[0] - r * (1, 0, -1, 0)[q]) < 1e-15 * max(r, 1) and abs(z1[0] - r * (0, 1, 0, -1)[q]) < 1e-15 * max(r, 1)
