"""The library's device-side random draws, restated in numpy (include/takzero_b200.h, "Device draws").

Every draw is rng_hash(seed, a, b, c) of the global game id a = game_base + g and a per-draw (b, c).  rng_hash takes
Python ints or numpy arrays (broadcast, uint64 arithmetic modulo 2^64) and returns an int for scalar arguments.

Counters of a handle, as api.cu keeps them: `move_counter` starts at 0 and goes up by one at the end of every device
search; a search's noise uses the counter before it, tz_select_selfplay and the sample inside tz_selfplay_move the
counter after it.  `opening_counter` goes up by one on every tz_new_openings and every restart, whether or not a game
finished.  Random steps are keyed by the ply alone."""
import numpy as np

GUMBEL_BITS = 23  # the field of h that makes the Gumbel uniform
SAMPLE_KEY = 0x5E1EC
OPENING_KEY = 0x0FE11
RANDOM_STEP_KEY = 0x57E95


def _u64(x):
    return np.asarray(x, dtype=np.uint64)


def mix64(x):
    with np.errstate(over="ignore"):
        x = _u64(x)
        x = x ^ (x >> np.uint64(33))
        x = x * np.uint64(0xFF51AFD7ED558CCD)
        x = x ^ (x >> np.uint64(33))
        x = x * np.uint64(0xC4CEB9FE1A85EC53)
        return x ^ (x >> np.uint64(33))


def rng_hash(seed, a, b, c):
    with np.errstate(over="ignore"):
        h = mix64(_u64(seed) ^ np.uint64(0x9E3779B97F4A7C15))
        h = mix64(h ^ (_u64(a) * np.uint64(0xBF58476D1CE4E5B9)))
        h = mix64(h ^ (_u64(b) * np.uint64(0x94D049BB133111EB)))
        h = mix64(h ^ (_u64(c) * np.uint64(0xD6E8FEB86659FD93)))
    return int(h) if h.ndim == 0 else h


# ---- Gumbel noise (k_gumbel_noise): one draw per (game, child index i) -------------------------------------------

def gumbel_field(seed, a, counter, i, bits=GUMBEL_BITS):
    """The top `bits` bits of rng_hash(seed, a, counter, i)."""
    return _u64(rng_hash(seed, a, counter, i)) >> np.uint64(64 - bits)


def gumbel_uniform(x, bits=GUMBEL_BITS):
    """u = ((float)x + 0.5f) * 2^-bits, in float32 as the kernel computes it."""
    return (np.asarray(x).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -bits)


def _log_faithful(x):
    """(lo, hi): the float32 values within 1 ulp of ln(x) for float32 x > 0 -- the float32 neighbours of the float64
    logarithm, or the three floats around it when it is too close to a float32 for float64 to tell the side."""
    y = np.log(x.astype(np.float64))
    f = y.astype(np.float32)
    down, up = np.nextafter(f, np.float32(-np.inf)), np.nextafter(f, np.float32(np.inf))
    d = f.astype(np.float64) - y
    unsure = np.abs(d) <= 1e-14 * np.abs(y)
    return np.where(unsure | (d > 0), down, f), np.where(unsure | (d < 0), up, f)


def gumbel_noise_bounds(u):
    """(lo, hi): the interval the device's -logf(-logf(u)) lies in, for float32 u in (0, 1).

    Device logf is within 1 ulp of the exact logarithm: its float32 result is one of the two floats around it.  Step 1
    gives a = logf(u) in [a_lo, a_hi]; step 2 gives logf(-a) between the lower neighbour of ln(-a_hi) and the upper
    one of ln(-a_lo); the noise is its negation.  The interval is a few ulps of the values wide, so it stays tight
    where the noise is near 0, and tests/test_device_draws.py checks that it separates neighbouring u."""
    u = np.asarray(u, dtype=np.float32)
    a_lo, a_hi = _log_faithful(u)
    c_lo, _ = _log_faithful(-a_hi)
    _, c_hi = _log_faithful(-a_lo)
    return -c_hi, -c_lo


def gumbel_rows(seed, base, G, counter, stride):
    """Uniforms [G, stride] of games base .. base + G - 1 at `counter`, as tz_last_gumbel lays out the noise."""
    a = np.arange(base, base + G, dtype=np.uint64)[:, None]
    i = np.arange(stride, dtype=np.uint64)[None, :]
    return gumbel_uniform(gumbel_field(seed, a, counter, i))


# ---- the other draws ------------------------------------------------------------------------------------------

def sample_randoms(seed, base, G, counter):
    """The random of k_select_actions per game: the first child whose cumulative weight exceeds r mod total."""
    return _u64(rng_hash(seed, np.arange(base, base + G, dtype=np.uint64), counter, SAMPLE_KEY))


def opening_draws(seed, base, G, counter):
    """(sym, adj) of k_new_openings / k_restart per game: h & 7 and (h >> 3) & 1."""
    h = _u64(rng_hash(seed, np.arange(base, base + G, dtype=np.uint64), counter, OPENING_KEY))
    return (h & np.uint64(7)).astype(np.int32), ((h >> np.uint64(3)) & np.uint64(1)).astype(np.int32)


def random_step_index(seed, a, ply, count):
    """Index into the legal moves (in possible_moves order) of the random step at `ply` of game a."""
    return rng_hash(seed, a, ply, RANDOM_STEP_KEY) % count


# ---- planted keys: game ids whose first draw (seed 7, counter 0, child 0) hits an edge of the field -----------------
# tests/test_device_draws.py re-derives each as the first game id from 0 on with that field value.

PLANT_SEED = 7
PLANTED = {  # name: (game id, field value)
    "bottom": (7295257, 0),
    "below_half": (2884750, (1 << 22) - 1),
    "half": (2474608, 1 << 22),  # 2^(bits-1): where a 24-bit field's x + 0.5f started to round
    "above_half": (7521953, (1 << 22) + 1),
    "top": (11284203, (1 << 23) - 1),  # also the top of a 24-bit field, where u rounded to 1.0f and the noise was +inf
}
