"""The device's Gumbel uniform and transform (k_gumbel_noise), restated in float32 as the kernel computes them and
checked at every value of the field; the planted game ids of tests/test_gpu_device_draws.py, re-derived."""
import numpy as np

from draws import (GUMBEL_BITS, PLANT_SEED, PLANTED, gumbel_field, gumbel_noise_bounds, gumbel_uniform, rng_hash)


def uniform_defects(bits: int) -> list:
    """What is wrong with u = ((float)x + 0.5f) * 2^-bits over all 2^bits field values x (empty: nothing)."""
    x = np.arange(1 << bits, dtype=np.uint32)
    u = gumbel_uniform(x, bits)
    defects = []
    if not np.array_equal(u.astype(np.float64), (x.astype(np.float64) + 0.5) * 2.0 ** -bits):
        defects.append("u is not (x + 1/2) * 2^-bits")
    if not ((u > 0) & (u < 1)).all():
        defects.append("u outside (0, 1)")
    if not (np.diff(u) > 0).all():
        defects.append("two field values give the same u")
    with np.errstate(divide="ignore"):
        noise = -np.log(-np.log(u))
    if not np.isfinite(noise).all():
        defects.append("non-finite noise")
    return defects


def test_the_uniform_is_exact_distinct_and_inside_the_open_interval():
    assert uniform_defects(GUMBEL_BITS) == []
    top = gumbel_uniform((1 << GUMBEL_BITS) - 1)
    assert top == np.float32(1.0 - 2.0 ** -24) and top < 1


def test_a_24_bit_field_fails_the_same_check():
    """The earlier formula, ((float)(h >> 40) + 0.5f) * 2^-24: x + 0.5f rounds to even above 2^23, the top value
    gives u = 1.0f and the noise -log(-log 1) = +inf."""
    defects = set(uniform_defects(24))
    assert defects == {"u is not (x + 1/2) * 2^-bits", "u outside (0, 1)", "two field values give the same u",
                       "non-finite noise"}
    u = gumbel_uniform(np.arange(1 << 24, dtype=np.uint32), 24)
    assert u[-1] == np.float32(1.0)
    with np.errstate(divide="ignore"):
        assert -np.log(-np.log(u[-1])) == np.inf
    assert len(np.unique(u[1 << 23:])) == (1 << 22) + 1  # the upper half: 2^23 inputs, 2^22 + 1 values


def test_the_noise_bounds_separate_neighbouring_uniforms():
    """The error model of the GPU tests: each interval holds the float64 value and lies strictly below the next
    field value's, so a device noise inside the interval of the restated u also pins u itself, bit for bit."""
    x = np.arange(1 << GUMBEL_BITS, dtype=np.uint32)
    u = gumbel_uniform(x)
    lo, hi = gumbel_noise_bounds(u)
    exact = -np.log(-np.log(u.astype(np.float64)))
    assert np.isfinite(lo).all() and np.isfinite(hi).all()
    assert (lo <= exact).all() and (exact <= hi).all()
    assert (hi[:-1] < lo[1:]).all()
    # the bound is relative to the values' ulps, not a flat tolerance: near 0 it is far below 1e-6
    near0 = np.abs(exact) < 1e-3
    assert near0.any() and (hi - lo)[near0].max() < 1e-6


def test_the_planted_game_ids_are_the_first_with_their_field_values():
    """By a search over game ids 0, 1, 2, ..: seed 7, counter 0 (the first search of a handle), child 0."""
    want = {name: value for name, (_, value) in PLANTED.items()}
    first = {}
    chunk = 1 << 21
    for lo in range(0, 1 << 25, chunk):
        field = gumbel_field(PLANT_SEED, np.arange(lo, lo + chunk, dtype=np.uint64), 0, 0)
        for name, value in want.items():
            hit = np.flatnonzero(field == value)
            if name not in first and len(hit):
                first[name] = lo + int(hit[0])
        if len(first) == len(want):
            break
    assert first == {name: gid for name, (gid, _) in PLANTED.items()}


def test_the_top_key_was_the_top_of_the_24_bit_field():
    gid = PLANTED["top"][0]
    h = rng_hash(PLANT_SEED, gid, 0, 0)
    assert h >> 40 == (1 << 24) - 1
    assert gumbel_uniform(h >> 40, 24) == np.float32(1.0)
    assert gumbel_uniform(h >> 41) == np.float32(1.0 - 2.0 ** -24)
    lo, hi = gumbel_noise_bounds(gumbel_uniform(h >> 41))
    assert 16.5 < lo <= hi < 16.7

