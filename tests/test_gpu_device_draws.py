"""GPU: every draw the library makes on the device equals its restatement in tests/draws.py.

Gumbel noise through tz_gumbel_sequential_halving (gumbel = NULL), tz_selfplay_move and tz_reanalyze_batch, read
back with tz_last_gumbel, must lie in the interval of the stated error model around the restated uniform (device logf
is within 1 ulp; the interval separates neighbouring uniforms, so it pins the uniform bit for bit).  The self-play
sample, the openings of tz_new_openings and of every restart, and tz_random_steps must equal the oracle or the
explicit-argument calls driven by the restated draws.  Game ids planted with game_base on the edges of the uniform's
field check the noise where the earlier 24-bit uniform returned +inf."""
import numpy as np
import pytest

from draws import (PLANT_SEED, PLANTED, gumbel_noise_bounds, gumbel_rows, gumbel_uniform, opening_draws,
                   random_step_index, sample_randoms)
from helpers import assert_roots_equal, games_to_states, state_to_game, states_equal
from oracle import oracle as O
from takzero_b200 import capi

pytestmark = pytest.mark.gpu

HK = 4
ENTRIES = ("gumbel", "selfplay", "reanalyze")
INT_MAX = 2**31 - 1


@pytest.fixture(autouse=True)
def _device_matching_math():
    O.lib().tk_set_exact_math(1)
    yield
    O.lib().tk_set_exact_math(0)


def selfplay_params(k, budget, seed, plies=10, threshold=32):
    return capi.SelfplayParams(k, budget, 0.0, plies, threshold, 0.5, float(budget), 0.25, seed)


def search(m, entry, k, budget, seed):
    """One device search with device-drawn noise through `entry`."""
    if entry == "gumbel":
        m.gumbel_sequential_halving(None, k, budget, None, seed=seed)
    elif entry == "selfplay":
        m.selfplay_move(selfplay_params(k, budget, seed, threshold=2))  # threshold 2: the early plies do sample
    else:
        m.reanalyze_batch(None, capi.ReanalyzeParams(k, budget, 0.25, seed))


def check_noise(m, seed, counter, what=""):
    """The noise of the last search against the restated draws of `counter`; returns it."""
    noise = m.last_gumbel()
    u = gumbel_rows(seed, m.game_base, m.G, counter, m.move_stride)
    lo, hi = gumbel_noise_bounds(u)
    assert np.isfinite(noise).all(), f"{what}: non-finite noise at (game, child) {np.argwhere(~np.isfinite(noise))[0]}"
    bad = np.argwhere((noise < lo) | (noise > hi))
    assert len(bad) == 0, (f"{what}: {len(bad)} draws outside the error model, first (game, child) {bad[0]}: "
                           f"{noise[tuple(bad[0])]!r} not in [{lo[tuple(bad[0])]!r}, {hi[tuple(bad[0])]!r}]")
    return noise


def opening_states(n, sym, adj):
    return games_to_states([O.new_opening(n, HK, int(s), int(a)) for s, a in zip(sym, adj)])


def assert_positions(got, want, what):
    for g in range(len(want)):
        assert states_equal(got[g], want[g]), f"{what}: game {g}"


# ---- Gumbel noise ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("n,G,base", [(3, 7, 0), (4, 5, 1000), (5, 13, 77), (6, 3, INT_MAX - 3)])
def test_device_noise_is_the_restated_draw(entry, n, G, base):
    """The first search of a handle draws at counter 0, each later one at the next counter; default strides, G not a
    multiple of 4 games per CTA or of the noise kernel's 256 threads, and game ids up to INT_MAX - 1."""
    m = capi.BatchedMCTS(n, HK, G, game_base=base, arena_slots=1 << 14)
    m.new_openings(seed=1)
    for counter in range(3):
        search(m, entry, 4, 8, seed=11)
        check_noise(m, 11, counter, f"{entry} search {counter}")
    assert m.status() == 0
    m.close()


def test_counters_across_a_mixed_sequence():
    """Both counters on one handle through every call that advances them: a search with injected noise advances the
    move counter too, a restart advances the opening counter when no game finished."""
    n, G, base, seed = 4, 6, 40, 5
    m = capi.BatchedMCTS(n, HK, G, game_base=base, arena_slots=1 << 15)
    mc = oc = 0

    def openings_at(counter, what):
        assert_positions(m.positions(), opening_states(n, *opening_draws(seed, base, G, counter)), what)

    m.new_openings(seed=seed)
    openings_at(oc, "first openings")
    oc += 1
    for step in range(2):
        m.gumbel_sequential_halving(None, 4, 8, None, seed=seed)
        check_noise(m, seed, mc, f"round {step}: search")
        mc += 1
        m.selfplay_move(selfplay_params(4, 8, seed))
        check_noise(m, seed, mc, f"round {step}: selfplay move")
        mc += 1
        oc += 1
        assert (m.restart_terminal_envs(seed=seed) == 0).all()  # nothing finished this early
        oc += 1
        m.reanalyze_batch(None, capi.ReanalyzeParams(4, 8, 0.25, seed))
        check_noise(m, seed, mc, f"round {step}: reanalyze")
        mc += 1
        m.gumbel_sequential_halving(None, 4, 8, np.zeros((G, m.move_stride), np.float32))
        mc += 1
        m.new_openings(seed=seed)
        openings_at(oc, f"round {step}: openings")
        oc += 1
    m.gumbel_sequential_halving(None, 4, 8, None, seed=seed)
    check_noise(m, seed, mc, "last search")
    assert m.status() == 0
    m.close()


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("G,offset", [(1, 0), (5, 2)])
@pytest.mark.parametrize("key", sorted(PLANTED))
def test_planted_keys(key, G, offset, entry):
    """A game on each planted id (seed 7, first search, child 0): finite noise, the restated value, and the search
    fed the read-back noise equals the oracle root for root with the same selected moves."""
    gid, field = PLANTED[key]
    n, k, budget = 4, 8, 48
    m = capi.BatchedMCTS(n, HK, G, game_base=gid - offset, arena_slots=1 << 15)
    m.new_openings(seed=3)
    start = m.positions()
    if entry == "gumbel":
        got = m.gumbel_sequential_halving(np.zeros(G, np.float32), k, budget, None, seed=PLANT_SEED)
    else:
        search(m, entry, k, budget, PLANT_SEED)
    noise = check_noise(m, PLANT_SEED, 0, key)
    lo, hi = gumbel_noise_bounds(gumbel_uniform(field))
    assert lo <= noise[offset, 0] <= hi
    if entry == "selfplay":  # the roots moved on; the other two leave the searched roots in place
        m.close()
        return
    ob = O.Batched([state_to_game(s, n, HK) for s in start])
    want = ob.gumbel_sequential_halving("synthetic", [0.0] * G, k, budget, noise)
    if entry == "gumbel":
        assert list(got) == want
    assert_roots_equal(m, ob, f"{key} {entry}")  # reanalyze: the roots its value targets are taken from
    m.close()


@pytest.mark.parametrize("entry", ENTRIES)
def test_sharded_draws_equal_unsharded(entry):
    """Handles over games [0, G/2) and [G/2, G) draw, concatenated, what one handle over [0, G) draws: noise bit for
    bit, openings, and (self-play) the sampled moves and the restarts, move after move."""
    n, G, seed = 3, 10, 9
    full = capi.BatchedMCTS(n, HK, G, arena_slots=1 << 15)
    halves = [capi.BatchedMCTS(n, HK, G // 2, game_base=b, arena_slots=1 << 15) for b in (0, G // 2)]
    handles = [full] + halves
    for m in handles:
        m.new_openings(seed=seed)
    cat = lambda f: np.concatenate([f(h) for h in halves])
    assert full.positions().tobytes() == cat(lambda h: h.positions()).tobytes()
    for step in range(12 if entry == "selfplay" else 3):
        for m in handles:
            search(m, entry, 4, 16, seed)
        assert np.array_equal(full.last_gumbel().view(np.uint32), cat(lambda h: h.last_gumbel()).view(np.uint32))
        if entry == "gumbel":
            sel = lambda h: h.select_actions_in_selfplay(10, 4, 0.5, None, seed=seed)
            assert np.array_equal(sel(full), cat(sel)), f"step {step}: sampled moves"
        assert full.positions().tobytes() == cat(lambda h: h.positions()).tobytes(), f"step {step}: positions"
    for m in handles:
        m.close()


# ---- self-play sampling ------------------------------------------------------------------------------------------

def test_selfplay_sample_equals_the_oracle_with_the_restated_random():
    """tz_select_selfplay(randoms = NULL) after a device search = tk_node_select_selfplay_action with the restated
    random of the counter after the search, per game.  3x3 positions where the visit threshold, the allowed eval drop
    and the proven-win filter each drop visited children, and positions past weighted_random_plies."""
    n, hk, G, k, budget, wrp, thr, drop, seed, base = 3, 0, 46, 8, 96, 10, 8, 0.1, 21, 500
    d = O.playout_positions(n, hk, 31, 1, 3000)
    st = d["states"].view(capi.STATE_DTYPE).reshape(-1)
    live = np.flatnonzero(d["terminal"] == 0)
    rng = np.random.default_rng(0)
    early, late = live[st["ply"][live] < wrp], live[st["ply"][live] >= wrp]
    pick = np.concatenate([rng.choice(early, G - 6, replace=False), rng.choice(late, 6, replace=False)])
    games = [d["games"][int(i)].copy() for i in pick]
    m = capi.BatchedMCTS(n, hk, G, game_base=base, arena_slots=1 << 15)
    m.set_positions(games_to_states(games))
    m.gumbel_sequential_halving(None, k, budget, None, seed=seed)
    noise = check_noise(m, seed, 0)
    ob = O.Batched(games)
    ob.gumbel_sequential_halving("synthetic", [0.0] * G, k, budget, noise)
    assert_roots_equal(m, ob, "search")
    got = m.select_actions_in_selfplay(wrp, thr, drop, None, seed=seed)
    r = sample_randoms(seed, base, G, 1)
    L = O.lib()
    dropped = {"threshold": 0, "win": 0, "eval drop": 0}
    for g in range(G):
        node = ob.node(g)
        sample = games[g].ply < wrp
        want = L.tk_node_select_selfplay_action(ob.node_ptr(g), int(sample), thr, drop, int(r[g]))
        assert got[g] == want, f"game {g}"
        if not sample or node.evaluation.tag != O.E_VALUE:
            continue
        ch = [node.children[i] for i in range(node.n_children)]
        best = ch[0].evaluation
        for c in ch[1:]:
            best = c.evaluation if L.tk_eval_cmp(c.evaluation, best) < 0 else best
        limit = O.make_eval(best.tag, best.u.value + np.float32(drop) if best.tag == O.E_VALUE else best.u.ply)
        for c in ch:
            if 0 < c.visit_count < thr:
                dropped["threshold"] += 1
            elif c.visit_count >= thr and c.evaluation.tag == O.E_WIN:
                dropped["win"] += 1
            elif c.visit_count >= thr and L.tk_eval_cmp(c.evaluation, limit) > 0:
                dropped["eval drop"] += 1
    assert min(dropped.values()) > 0, dropped
    m.close()


def test_selfplay_move_equals_the_host_sequence_driven_by_the_restated_draws():
    """tz_selfplay_move with recording on: noise at counter c, the sample at c + 1, the restart's openings at the
    opening counter.  A second handle runs the host-buffer calls with all three injected (the read-back noise after it
    is checked against the restatement, the sample randoms and openings restated) and must play the same moves."""
    n, G, k, budget, wrp, seed, base = 3, 12, 4, 16, 10, 3, 90
    sp = selfplay_params(k, budget, seed, plies=wrp, threshold=2)
    a = capi.BatchedMCTS(n, HK, G, game_base=base, arena_slots=1 << 15)
    b = capi.BatchedMCTS(n, HK, G, arena_slots=1 << 15)
    a.new_openings(seed=seed)
    b.set_positions(a.positions())
    a.selfplay_record(True)
    finished = 0
    for c in range(40):
        a.selfplay_move(sp)
        noise = check_noise(a, seed, c, f"move {c}")
        cur = b.positions()
        selected = b.gumbel_sequential_halving(np.zeros(G, np.float32), k, budget, noise)
        sampled = b.select_actions_in_selfplay(wrp, 2, 0.5, sample_randoms(seed, base, G, c + 1))
        b.step(np.where(cur["ply"] < wrp, sampled, selected).astype(np.uint16))
        term = b.restart_terminal_envs(*opening_draws(seed, base, G, 1 + c))
        assert a.positions().tobytes() == b.positions().tobytes(), f"move {c}"
        rec = a.selfplay_read()
        assert sorted(rec["replay_game"] - base) == list(np.flatnonzero(term)), f"move {c}: finished games"
        for j in range(rec["n_replays"]):
            o, length = int(rec["replay_offset"][j]), int(rec["replay_length"][j])
            _, moves = b.finished_replay(int(rec["replay_game"][j]) - base)
            assert np.array_equal(rec["replay_moves"][o:o + length], moves), f"move {c}: replay {j}"
        finished += rec["n_replays"]
    assert finished >= 5 and a.status() == 0 and b.status() == 0
    a.close()
    b.close()


# ---- openings, restarts, random steps ----------------------------------------------------------------------------

def test_openings_and_restarts_are_the_restated_draws():
    n, hk, G, seed, base = 3, 0, 14, 12, 321
    m = capi.BatchedMCTS(n, hk, G, game_base=base, arena_slots=1 << 14)
    for oc in range(2):
        m.new_openings(seed=seed)
        sym, adj = opening_draws(seed, base, G, oc)
        want = games_to_states([O.new_opening(n, hk, int(s), int(a)) for s, a in zip(sym, adj)])
        assert_positions(m.positions(), want, f"new_openings {oc}")
    d = O.playout_positions(n, hk, 8, 1, 2000)
    st = d["states"].view(capi.STATE_DTYPE).reshape(-1)
    live, done = np.flatnonzero(d["terminal"] == 0), np.flatnonzero(d["terminal"] != 0)
    rng = np.random.default_rng(1)
    m.set_positions(st[rng.choice(live, G, replace=False)])
    before = m.positions()
    assert (m.restart_terminal_envs(seed=seed) == 0).all()  # opening counter 2, nothing restarts
    assert m.positions().tobytes() == before.tobytes()
    mixed = st[rng.choice(live, G, replace=False)].copy()
    ended = np.arange(G) % 3 == 1
    mixed[ended] = st[rng.choice(done, int(ended.sum()), replace=False)]
    m.set_positions(mixed)
    term = m.restart_terminal_envs(seed=seed)  # opening counter 3
    assert np.array_equal(term != 0, ended)
    sym, adj = opening_draws(seed, base, G, 3)
    want = mixed.copy()
    want[ended] = games_to_states([O.new_opening(n, hk, int(sym[g]), int(adj[g])) for g in np.flatnonzero(ended)])
    assert_positions(m.positions(), want, "restart")
    m.close()


@pytest.mark.parametrize("n,G,steps", [(3, 9, 40), (5, 6, 12)])
def test_random_steps_are_the_restated_draws(n, G, steps):
    """moves[h mod count] in possible_moves order, keyed by the ply, stopping at a finished game."""
    seed, base = 17, 2024
    m = capi.BatchedMCTS(n, HK, G, game_base=base, arena_slots=1 << 14)
    m.new_openings(seed=seed)
    start = m.positions()
    m.random_steps(steps, seed=seed)
    got = m.positions()
    stopped = 0
    for g in range(G):
        game = state_to_game(start[g], n, HK)
        for _ in range(steps):
            if O.terminal(game) != O.T_NONE:
                stopped += 1
                break
            moves = O.possible_moves(game)
            O.play(game, moves[random_step_index(seed, base + g, game.ply, len(moves))])
        assert states_equal(got[g], games_to_states([game])[0]), f"game {g}"
    if n == 3:
        assert stopped > 0, "some games end within the steps"
    m.close()
