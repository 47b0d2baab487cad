"""GPU parity: the batched search through the C ABI vs the CPU oracle, bit-exact.

With identical agent outputs (the integer-hash synthetic agent on both sides, or the oracle's
agents injected through the host callback) and identical injected Gumbel noise / openings,
visit counts, evaluations (f32 bits), priors, selected moves, targets and replays must be
identical to the restated reference (takzero/src/search/node/{mcts,batched,policy,mod}.rs)."""
import numpy as np
import pytest

from oracle import oracle as O
from takzero_b200 import capi

from helpers import (assert_roots_equal, games_to_states, host_agent_from_oracle, random_playout_states,
                     states_equal)

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _device_matching_math():
    O.lib().tk_set_exact_math(1)
    yield
    O.lib().tk_set_exact_math(0)


def make_pair(n, half_komi, G, seed, arena_slots=1 << 15, from_playouts=False):
    rng = np.random.default_rng(seed)
    if from_playouts:
        games = []
        while len(games) < G:
            ps = [p for p in random_playout_states(n, half_komi, int(rng.integers(1 << 30)), keep_terminal=False)]
            games.append(ps[int(rng.integers(len(ps)))])
    else:
        games = [O.new_opening(n, half_komi, int(rng.integers(8)), int(rng.integers(2))) for _ in range(G)]
    ob = O.Batched(games)
    m = capi.BatchedMCTS(n, half_komi, G, arena_slots=arena_slots)
    m.set_positions(games_to_states(games))
    return m, ob, rng


@pytest.mark.parametrize("n,half_komi,G,sims", [(3, 0, 16, 300), (4, 4, 32, 120), (5, 4, 16, 80), (6, 4, 16, 60)])
def test_simulate_synthetic(n, half_komi, G, sims):
    m, ob, rng = make_pair(n, half_komi, G, 100 + n)
    betas = rng.random(G).astype(np.float32) * 0.5
    for s in range(sims):
        m.simulate(betas)
        ob.simulate("synthetic", betas)
        if s in (0, 1, 5, sims // 2):
            assert_roots_equal(m, ob, f"after sim {s}")
    assert_roots_equal(m, ob, "final")
    c, oc = m.counters(), ob.counters()
    assert (c.simulations, c.evaluations, c.known) == (oc.simulations, oc.evaluations, oc.known)
    m.close()


@pytest.mark.parametrize("agent", ["simple", "dummy"])
def test_simulate_injected_agent(agent):
    """Reference agents `Dummy` / `Simple` (agent.rs:16-87) injected through the host callback."""
    n, hk, G = 4, 4, 8
    m, ob, rng = make_pair(n, hk, G, 7, from_playouts=True)
    cb = host_agent_from_oracle(agent, n, hk)
    m.set_agent(capi.AGENT_HOST, cb)
    betas = np.zeros(G, dtype=np.float32)
    for s in range(150):
        m.simulate(betas)
        ob.simulate(agent, betas)
    assert_roots_equal(m, ob, agent)
    m.close()


def test_solver_finds_tinue():
    """mcts.rs:345-376 `find_tinue_easy` on the GPU trees (Dummy agent, beta = 1... here 0)."""
    g = O.from_ptn_moves(3, 0, ["a3", "c1", "c2", "c3", "b3", "c3-"])
    G = 4
    m = capi.BatchedMCTS(3, 0, G, arena_slots=1 << 16)
    m.set_positions(games_to_states([g] * G))
    m.set_agent(capi.AGENT_HOST, host_agent_from_oracle("dummy", 3, 0))
    ob = O.Batched([g] * G)
    betas = np.ones(G, dtype=np.float32)
    solved = False
    for s in range(5000):
        m.simulate(betas)
        ob.simulate("dummy", betas)
        if s % 50 == 49:
            st = m.root_stats()
            if (st["eval_tag"] == capi.E_WIN).all():
                solved = True
                break
    assert solved
    assert_roots_equal(m, ob, "tinue")
    tbl = m.root_children()
    loss = [i for i in range(tbl["n"][0]) if tbl["eval_tag"][0, i] == capi.E_LOSS]
    assert [O.move_str(int(tbl["moves"][0, i])) for i in loss] == ["b1"]
    assert O.move_str(int(m.select_best_actions()[0])) == "b1"
    m.close()


def run_selfplay_pair(n, half_komi, G, k, budget, moves, seed, agent="synthetic", games=None):
    if games is None:
        m, ob, rng = make_pair(n, half_komi, G, seed)
    else:
        rng = np.random.default_rng(seed)
        ob = O.Batched(games)
        m = capi.BatchedMCTS(n, half_komi, G, arena_slots=1 << 16)
        m.set_positions(games_to_states(games))
    if agent != "synthetic":
        m.set_agent(capi.AGENT_HOST, host_agent_from_oracle(agent, n, half_komi))
    stride = m.move_stride
    finished = 0
    for mv in range(moves):
        betas = (rng.random(G) < 0.5).astype(np.float32) * 0.25
        gumbel = rng.gumbel(size=(G, stride)).astype(np.float32)
        got = m.gumbel_sequential_halving(betas, k, budget, gumbel)
        want = ob.gumbel_sequential_halving(agent, betas, k, budget, gumbel)
        assert list(got) == want, f"move {mv}: selected actions"
        assert_roots_equal(m, ob, f"move {mv} after search")
        # targets (selfplay/src/main.rs:243-256): improved policy + ube target
        vis = float((budget // int(np.log2(k)) // k) * (k - 1))
        pol, ube, cnt = m.targets(vis, 0.25)
        for g in range(G):
            node = ob.node_ptr(g)
            want_pol = O.improved_policy(node, vis)
            assert cnt[g] == len(want_pol)
            assert np.array_equal(pol[g, : cnt[g]].view(np.uint32), want_pol.view(np.uint32)), f"move {mv} game {g}: improved policy"
            want_ube = O.lib().tk_node_ube_target(node, 0.25)
            assert np.float32(ube[g]).view(np.uint32) == np.float32(want_ube).view(np.uint32)
        # early plies: visit-weighted sampling with injected randomness (node/mod.rs:170-207)
        randoms = rng.integers(0, 1 << 62, size=G, dtype=np.uint64)
        sel = m.select_actions_in_selfplay(10, 8, 0.5, randoms)
        for g in range(G):
            env = ob.env(g)
            w = O.lib().tk_node_select_selfplay_action(ob.node_ptr(g), int(env.ply < 10), 8, 0.5, int(randoms[g]))
            assert sel[g] == w, f"move {mv} game {g}: selfplay action"
        best = m.select_best_actions()
        assert list(best) == ob.select_best_actions()
        play = np.where(np.arange(G) % 2 == 0, got, sel).astype(np.uint16)
        m.step(play)
        ob.step([int(x) for x in play])
        assert_roots_equal(m, ob, f"move {mv} after step")
        sym = rng.integers(0, 8, size=G).astype(np.int32)
        adj = rng.integers(0, 2, size=G).astype(np.int32)
        term = m.restart_terminal_envs(sym, adj)
        replays_before = [ob.replay(g) for g in range(G)]
        want_term = ob.restart_terminal_envs([int(x) for x in sym], [int(x) for x in adj])
        assert list(term) == want_term
        for g in range(G):
            if term[g] != capi.T_NONE:
                finished += 1
                _, mv_list = m.finished_replay(g)
                assert list(mv_list) == replays_before[g]
        pos = m.positions()
        want_pos = games_to_states([ob.env(g) for g in range(G)])
        for g in range(G):
            assert states_equal(pos[g], want_pos[g]), f"move {mv} game {g}: env"
            _, cur = m.replay(g)
            assert list(cur) == ob.replay(g)
    c, oc = m.counters(), ob.counters()
    assert (c.simulations, c.evaluations, c.known) == (oc.simulations, oc.evaluations, oc.known)
    m.close()
    return finished


def test_gumbel_selfplay_4x4():
    finished = run_selfplay_pair(4, 4, 24, 16, 64, 40, seed=1)
    assert finished > 0  # games ended and restarted inside the run


def test_gumbel_selfplay_3x3_long():
    finished = run_selfplay_pair(3, 0, 16, 4, 32, 40, seed=2)
    assert finished > 4


def test_gumbel_selfplay_5x5():
    run_selfplay_pair(5, 4, 8, 16, 64, 6, seed=3)


def test_gumbel_selfplay_6x6():
    run_selfplay_pair(6, 4, 8, 16, 128, 4, seed=4)


def test_gumbel_selfplay_6x6_full_budget_with_restarts():
    """BASELINE configs[2]'s search parameters (k = 16, 256 simulations per move) bit-exact over 12 moves, started
    from late-game 6x6 positions (boards with at most four empty squares) so that games end inside the run: roots,
    selected moves, targets, replays and the restarted positions all equal the oracle's."""
    n, hk, G = 6, 4, 12
    d = O.playout_positions(n, hk, 4242, 1, 40_000)
    st = d["states"].view(capi.STATE_DTYPE).reshape(-1)
    late = np.flatnonzero((d["terminal"] == 0) & ((st["height"][:, : n * n] == 0).sum(axis=1) <= 4))
    assert len(late) >= G
    picks = late[np.linspace(0, len(late) - 1, G).astype(int)]
    games = [d["games"][int(i)].copy() for i in picks]
    finished = run_selfplay_pair(n, hk, G, 16, 256, 12, seed=6, games=games)
    assert finished >= 3


def test_gumbel_selfplay_simple_agent():
    run_selfplay_pair(4, 4, 8, 8, 48, 12, seed=5, agent="simple")


def test_device_gumbel_noise_is_reproducible_and_injectable():
    """Library RNG mode: the noise it drew can be read back and injected into the oracle."""
    n, hk, G = 4, 4, 16
    m, ob, rng = make_pair(n, hk, G, 11)
    betas = np.zeros(G, dtype=np.float32)
    got = m.gumbel_sequential_halving(betas, 16, 64, None, seed=99)
    noise = m.last_gumbel()
    assert np.isfinite(noise).all() and noise.std() > 0.5
    want = ob.gumbel_sequential_halving("synthetic", betas, 16, 64, noise)
    assert list(got) == want
    assert_roots_equal(m, ob, "device noise")
    m.close()


def test_sharded_equals_unsharded():
    """Games are independent: two handles over halves of the batch == one handle (SURVEY 8e)."""
    n, hk, G = 4, 4, 16
    full = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    lo = capi.BatchedMCTS(n, hk, G // 2, game_base=0, arena_slots=1 << 14)
    hi = capi.BatchedMCTS(n, hk, G // 2, game_base=G // 2, arena_slots=1 << 14)
    for h in (full, lo, hi):
        h.new_openings(seed=5)
    moves_full = full.gumbel_sequential_halving(None, 8, 48, None, seed=7)
    moves = np.concatenate([lo.gumbel_sequential_halving(None, 8, 48, None, seed=7),
                            hi.gumbel_sequential_halving(None, 8, 48, None, seed=7)])
    assert np.array_equal(moves_full, moves)
    a = full.root_children()
    b0, b1 = lo.root_children(), hi.root_children()
    assert np.array_equal(a["visits"], np.concatenate([b0["visits"], b1["visits"]]))
    for h in (full, lo, hi):
        h.close()


def test_argument_errors():
    m = capi.BatchedMCTS(4, 4, 4, arena_slots=4096)
    m.new_openings(seed=1)
    with pytest.raises(capi.TakzeroError, match="multiple of k"):
        m.gumbel_sequential_halving(None, 16, 100, None)  # batched.rs:216-220
    with pytest.raises(capi.TakzeroError):
        m.gumbel_sequential_halving(None, 0, 64, None)  # batched.rs:215
    with pytest.raises(capi.TakzeroError, match="tz_set_weights"):
        m.set_agent(capi.AGENT_NETWORK)
    m.close()
    # game ids game_base + g key every device draw and must fit an int
    for base in (-1, 2**31 - 4, 2**31 - 1):
        with pytest.raises(capi.TakzeroError, match="game_base"):
            capi.BatchedMCTS(4, 4, 4, game_base=base, arena_slots=4096)
    capi.BatchedMCTS(4, 4, 4, game_base=2**31 - 5, arena_slots=4096).close()


def test_arena_overflow_is_reported():
    m = capi.BatchedMCTS(5, 4, 4, arena_slots=256)
    m.new_openings(seed=1)
    with pytest.raises(capi.TakzeroError, match="arena_full"):
        for _ in range(20):
            m.simulate(None)
    m.close()


def test_apply_noise_keeps_distribution():
    """node/noise.rs:48-67 `distribution_stays_1_after_noise`: after mixing Dirichlet noise the priors still
    sum to 1 and logit = ln p; the mixed priors are what the next search uses."""
    n, hk, G = 4, 4, 8
    m = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    m.new_openings(seed=3)
    m.simulate(None)
    before = m.root_children()
    rng = np.random.default_rng(0)
    noise = np.zeros((G, m.move_stride), dtype=np.float32)
    for g in range(G):
        noise[g, : before["n"][g]] = rng.dirichlet([0.3] * int(before["n"][g]))
    m.apply_noise(noise, 0.25)
    after = m.root_children()
    for g in range(G):
        k = after["n"][g]
        p = after["prob"][g, :k]
        assert abs(float(p.sum()) - 1.0) < 1e-5
        want = before["prob"][g, :k] * np.float32(0.75) + noise[g, :k] * np.float32(0.25)
        assert np.array_equal(p, want.astype(np.float32))
        assert np.array_equal(after["logit"][g, :k], np.log(p, dtype=np.float32))
    m.simulate(None)  # still searchable
    m.close()


def test_move_stride_overflow_is_reported():
    """More legal moves than the configured row stride: reported (TZ_STATUS_TOO_MANY_MOVES), never truncated."""
    m = capi.BatchedMCTS(5, 4, 4, arena_slots=4096, move_stride=16)
    m.new_openings(seed=1)
    with pytest.raises(capi.TakzeroError, match="too_many_moves"):
        m.simulate(None)
    m.close()


def test_single_game_and_odd_batch_sizes():
    """Ragged sizes: 1 game and a game count that is not a multiple of the 4 games per CTA."""
    for G in (1, 7):
        m, ob, rng = make_pair(4, 4, G, 50 + G)
        gum = rng.gumbel(size=(G, m.move_stride)).astype(np.float32)
        got = m.gumbel_sequential_halving(np.zeros(G, np.float32), 4, 32, gum)
        want = ob.gumbel_sequential_halving("synthetic", [0.0] * G, 4, 32, gum)
        assert list(got) == want
        assert_roots_equal(m, ob, f"G={G}")
        m.close()


def test_nan_and_infinite_network_outputs_raise_the_nan_bit_without_faulting():
    """The reference panics on a NaN logit / value (net6_simhash.rs:304, NotNan).  Here the device raises
    TZ_STATUS_NAN and replaces the outputs by finite ones before anything enters a tree -- a NaN in the arena would
    derail the argmax / ranking code that indexes it (this used to end in a CUDA `misaligned address` fault)."""
    n, hk, G = 4, 4, 8
    m = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    calls = [0]

    def cb(ctx, batch, envs, actions, n_actions, stride, logits, values, variances):
        calls[0] += 1
        lg = np.ctypeslib.as_array(logits, shape=(batch, stride))
        lg[:] = 0.1
        if calls[0] >= 3:
            lg[0::2, 0] = np.nan
            lg[1::2, :] = np.inf
        np.ctypeslib.as_array(values, shape=(batch,))[:] = np.nan if calls[0] >= 5 else 0.2
        np.ctypeslib.as_array(variances, shape=(batch,))[:] = -1.0 if calls[0] >= 7 else 1.0

    m.set_agent(capi.AGENT_HOST, cb)
    m.new_openings(seed=1)
    with pytest.raises(capi.TakzeroError, match="nan"):
        m.gumbel_sequential_halving(None, 8, 24, None, seed=0)
    assert m.status() == 32  # TZ_STATUS_NAN only: no other invariant broke, no CUDA error
    assert calls[0] >= 20    # the search ran to the end
    tbl = m.root_children()
    assert np.isfinite(tbl["prob"]).all() and np.isfinite(tbl["logit"]).all() and np.isfinite(tbl["std_dev"]).all()
    m.close()


def test_nan_noise_and_betas_from_the_host_are_reported_not_fatal():
    """Injected Gumbel noise / betas are host data: a NaN in them must end in TZ_STATUS_NAN with a complete
    candidate set, not in colliding ranks and stale child indices."""
    n, hk, G = 4, 4, 8
    m = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    m.new_openings(seed=2)
    gumbel = np.random.default_rng(0).gumbel(size=(G, m.move_stride)).astype(np.float32)
    gumbel[::2, :6] = np.nan
    with pytest.raises(capi.TakzeroError, match="nan"):
        m.gumbel_sequential_halving(None, 8, 24, gumbel)
    assert m.status() == 32
    m.close()
    m = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    m.new_openings(seed=2)
    betas = np.full(G, np.nan, dtype=np.float32)
    with pytest.raises(capi.TakzeroError, match="nan"):
        m.gumbel_sequential_halving(betas, 8, 24, None, seed=1)
    assert m.status() == 32
    m.close()


def test_invalid_move_in_step_is_reported():
    """`env.step(action)` with an illegal action: the reference panics ("Action should be valid", env.rs:44); here
    TZ_STATUS_BAD_MOVE is raised and the position is left alone."""
    n, hk, G = 4, 4, 4
    m = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 12)
    m.new_openings(seed=4)
    before = m.positions()
    moves = m.legal_moves(before)[0][:, 0].copy()
    moves[2] = 2 << 6  # Ca1: there are no capstones on 4x4
    m.simulate(None)
    roots_before = m.root_stats()
    try:
        m.step(moves)
    except capi.TakzeroError:
        pass
    assert m.status() == 16  # TZ_STATUS_BAD_MOVE
    after = m.positions()
    assert after[2].tobytes() == before[2].tobytes()           # the position of the offending game stays
    assert m.root_stats()[2] == roots_before[2]                  # and so does its tree
    assert after[0]["ply"] == before[0]["ply"] + 1             # the others moved on
    # an illegal spread that the move encoding allows (onto nothing, from an empty square) is refused by tz_apply too
    states, ok = m.apply(before, np.array([moves[0], 1 | (1 << 6) | (0x80 << 8), moves[2], moves[3]], dtype=np.uint16))
    assert list(ok) == [1, 0, 0, 1]
    assert states[1].tobytes() == before[1].tobytes() and states[2].tobytes() == before[2].tobytes()
    m.close()


def test_device_expf_is_the_restated_glibc_expf():
    """The softmax's exp on the device (tree.cuh `expf_libm`) against the oracle's `tk_expf_restated` -- the same
    glibc algorithm, which tests/test_oracle_golden.py shows equal to the host libm -- on 1.2*10^7 inputs: every
    8th f32 bit pattern of the softmax range [-104, 0] plus a sweep of the positive range.  Bit-exact."""
    import ctypes as C

    from takzero_b200 import network

    network._declare()
    L = capi.lib()
    m = capi.BatchedMCTS(4, 4, 4, arena_slots=4096)
    lo, hi = int(np.float32(-1e-30).view(np.uint32)), int(np.float32(-104.0).view(np.uint32))
    neg = np.arange(lo, hi, 41, dtype=np.uint32).view(np.float32)
    pos = np.arange(0, int(np.float32(89.0).view(np.uint32)), 257, dtype=np.uint32).view(np.float32)
    special = np.array([0.0, -0.0, np.inf, -np.inf, 88.72284, 88.72283, -103.97208, -103.972, np.nan], dtype=np.float32)
    xs = np.ascontiguousarray(np.concatenate([neg, pos, special]))
    assert len(xs) >= 12_000_000
    got = np.zeros_like(xs)
    want = np.zeros_like(xs)
    for a in range(0, len(xs), 1 << 22):
        chunk = np.ascontiguousarray(xs[a:a + (1 << 22)])
        out = np.zeros_like(chunk)
        assert L.tz_debug_expf(m.handle, chunk.ctypes.data, len(chunk), out.ctypes.data) == 0
        got[a:a + len(chunk)] = out
    O.lib().tk_expf_restated_batch(xs.ctypes.data, len(xs), want.ctypes.data)
    ok = (got.view(np.uint32) == want.view(np.uint32)) | (np.isnan(got) & np.isnan(want))
    assert ok.all(), f"{(~ok).sum()} mismatches, first at {xs[~ok][0]!r}"
    m.close()


def test_gumbel_rows_shorter_than_a_root_are_reported():
    """batched.rs:233-239 zips one Gumbel draw with every root child.  A caller whose noise rows are shorter than a
    root's child list has not supplied them: reported as TZ_STATUS_TOO_MANY_MOVES (never the next game's noise), the
    children without a draw rank last, and the search still ends with a complete candidate set."""
    n, hk, G = 4, 4, 8
    m = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    m.new_openings(seed=2)
    m.simulate(None)
    n_children = int(m.root_stats()["n_children"].min())
    assert n_children > 12
    gumbel = np.random.default_rng(0).gumbel(size=(G, 12)).astype(np.float32)
    with pytest.raises(capi.TakzeroError, match="too_many_moves"):
        m.gumbel_sequential_halving(None, 8, 24, gumbel)
    assert m.status() == 8
    m.close()
    # with rows as long as the longest child list the same call is fine
    m = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    m.new_openings(seed=2)
    m.simulate(None)
    width = int(m.root_stats()["n_children"].max())
    m.gumbel_sequential_halving(None, 8, 24, np.random.default_rng(0).gumbel(size=(G, width)).astype(np.float32))
    assert m.status() == 0
    m.close()


def test_reanalyze_batch_on_the_device_equals_the_host_loop():
    """reanalyze/src/main.rs:147-235 on the device (tz_stage_positions / tz_reanalyze_batch / tz_reanalyze_read): fresh
    roots picked out of a staged pool, search, then per root the improved policy at most_visited_count() visitations,
    the UBE target and the value target (root evaluation when known, else the negated evaluation of the selected
    child as f32).  Must equal, bit for bit, the same steps through the host-buffer calls with the value rule applied by
    the oracle's Eval functions."""
    n, hk, G, k, budget = 4, 4, 48, 8, 48
    rng = np.random.default_rng(21)
    d = O.playout_positions(n, hk, 5, 1, 4000)
    live = np.flatnonzero(d["terminal"] == 0)
    # late positions, so that some roots get solved and the "known root" branch of the value rule is exercised
    late = live[np.argsort(-d["states"].view(capi.STATE_DTYPE).reshape(-1)["ply"][live])[:300]]
    pool = d["states"].view(capi.STATE_DTYPE).reshape(-1)[late].copy()
    idx = rng.choice(len(pool), size=G, replace=False).astype(np.uint32)
    params = capi.ReanalyzeParams(k, budget, 0.25, 77)

    a = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    a.stage_positions(pool)
    a.reanalyze_batch(idx, params)
    got = a.reanalyze_read()
    assert a.status() == 0

    b = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    b.set_positions(pool[idx])
    selected = b.gumbel_sequential_halving(None, k, budget, None, seed=77)
    pol, ube, cnt, moves = b.targets(-1.0, 0.25, with_moves=True)
    roots, ch = b.root_stats(), b.root_children()
    L = O.lib()
    want_value = np.zeros(G, dtype=np.float32)
    solved = 0
    for g in range(G):
        if roots["eval_tag"][g] != capi.E_VALUE:
            e = O.make_eval(int(roots["eval_tag"][g]), int(roots["eval_bits"][g]))
            solved += 1
        else:
            i = int(np.flatnonzero(ch["moves"][g, : ch["n"][g]] == selected[g])[0])
            tag, bits = int(ch["eval_tag"][g, i]), int(ch["eval_bits"][g, i])
            child = O.make_eval(tag, bits if tag else float(np.uint32(bits).view(np.float32)))
            e = L.tk_eval_negate(child)
        want_value[g] = L.tk_eval_to_f32(e)
    assert solved > 0 and solved < G
    assert np.array_equal(got["n"], cnt)
    assert np.array_equal(got["moves"], moves)
    assert np.array_equal(got["policy"].view(np.uint32), pol.view(np.uint32))
    assert np.array_equal(got["ube"].view(np.uint32), ube.view(np.uint32))
    assert np.array_equal(got["value"].view(np.uint32), want_value.view(np.uint32))
    # a second batch on the same handle (other roots) and the error for an index outside the pool
    a.reanalyze_batch(rng.choice(len(pool), size=G, replace=False).astype(np.uint32), params)
    assert a.reanalyze_read()["n"].min() > 0 and a.status() == 0
    bad = idx.copy()
    bad[3] = len(pool)
    with pytest.raises(capi.TakzeroError, match="out of range"):
        a.reanalyze_batch(bad, params)
    for h in (a, b):
        h.close()
