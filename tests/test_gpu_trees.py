"""GPU: many single trees at once (tz_trees_simulate_batch / tz_trees_descend / tz_trees_principal_variation).

Every selected game's tree must come out exactly as the one-tree calls (tz_tree_*, game 0 of a handle of its own) leave
it when that tree is searched alone with the same moves: visits, evaluation tags and bits, priors, logits, standard
deviations and arena use of the root and its children, after every batch and every descend, and the same principal
variation.  The leaves of all trees share one network batch in an order that varies from run to run; a leaf's network
output does not depend on its row, so the trees do not either."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from takzero_b200 import capi, network, weights

from helpers import games_to_states, oracle_children, random_playout_states, state_to_game

pytestmark = pytest.mark.gpu

HK = 4
EXACT_KEYS = ("moves", "visits", "eval_tag", "eval_bits")
BIT_KEYS = ("logit", "prob", "std_dev")


@pytest.fixture(autouse=True)
def _device_matching_math():
    O.lib().tk_set_exact_math(1)
    yield
    O.lib().tk_set_exact_math(0)


def openings(n, count, seed, hk=HK):
    """`count` different seeded positions a few plies into random games (none terminal)."""
    out = []
    for t in range(count):
        line = random_playout_states(n, hk, 1000 * seed + t, max_plies=8, keep_terminal=False)
        out.append(line[min(len(line) - 1, t % 7)])
    return out


def snapshot(m, games):
    st, ch = m.root_stats(), m.root_children()
    return [(st[g].copy(), {k: ch[k][g].copy() for k in EXACT_KEYS + BIT_KEYS}) for g in games]


def assert_same_tree(a, b, what):
    (st_a, ch_a), (st_b, ch_b) = a, b
    for f in capi.ROOT_DTYPE.names:  # evaluation, visits, std, child count, arena use
        assert st_a[f] == st_b[f], f"{what}: root {f}"
    k = int(st_a["n_children"])
    for key in EXACT_KEYS:
        assert np.array_equal(ch_a[key][:k], ch_b[key][:k]), f"{what}: children {key}"
    for key in BIT_KEYS:
        assert np.array_equal(ch_a[key][:k].view(np.uint32), ch_b[key][:k].view(np.uint32)), f"{what}: children {key} bits"


def run_trees(m, plan, mask=None, pv_cap=16, seed=0):
    """Runs `plan` ([("sim", beta, batch) | ("descend",)]) on the selected trees of `m`.  At a descend, even trees play
    their best move (the PV's first), odd ones a visited sibling.  Returns one record per step: (step, moves, pvs,
    snapshots of the selected games)."""
    games = list(range(m.G)) if mask is None else [g for g in range(m.G) if mask[g]]
    rng = np.random.default_rng(seed)
    log = []
    for step in plan:
        moves = pv = None
        if step[0] == "sim":
            m.trees_simulate_batch(step[1], step[2], mask)
        else:
            pv = m.trees_principal_variation(pv_cap, mask)
            tbl = m.root_children()
            moves = np.zeros(m.G, np.uint16)
            for t, g in enumerate(games):
                assert pv[1][g] >= 1
                moves[g] = pv[0][g, 0]
                if t % 2:
                    visited = [int(tbl["moves"][g, i]) for i in range(tbl["n"][g]) if tbl["visits"][g, i] > 0]
                    moves[g] = visited[int(rng.integers(len(visited)))]
            m.trees_descend(moves, mask)
        log.append((step, moves, pv, snapshot(m, games)))
    return games, log


def replay_solo(s, state, t, g, log, what, pv_cap=16):
    """Tree t (game g of the many-tree handle; `state` [1]) searched alone on game 0 of handle `s`, step by step."""
    s.set_positions(state)
    for i, (step, moves, pv, snaps) in enumerate(log):
        if step[0] == "sim":
            s.tree_simulate_batch(step[1], step[2])
        else:
            assert list(s.tree_principal_variation(pv_cap)) == list(pv[0][g, :pv[1][g]]), f"{what} tree {t}: pv"
            s.tree_descend(int(moves[g]))
        assert_same_tree(snaps[t], snapshot(s, [0])[0], f"{what} tree {t} step {i} {step[0]}")


def counters_tuple(m):
    c = m.counters()
    return np.array([c.simulations, c.evaluations, c.known, c.expansions], np.uint64)


PLAN = ([("sim", 0.0, None)] * 3 + [("descend",)]) * 2 + [("sim", 0.0, None)] * 2 + [("sim", 0.5, None)]


@pytest.mark.parametrize("warps", [1, 8])
@pytest.mark.parametrize("trees", [2, 7, 32])
@pytest.mark.parametrize("n,batch", [(4, 16), (5, 24), (6, 32)])
def test_many_trees_equal_solo_trees(n, batch, trees, warps):
    states = games_to_states(openings(n, trees, seed=n))
    m = capi.BatchedMCTS(n, HK, trees, tree_batch=trees * batch, arena_slots=1 << 16)
    s = capi.BatchedMCTS(n, HK, 1, tree_batch=batch, arena_slots=1 << 16)
    for h in (m, s):
        h.debug_tree_warps(warps)
    m.set_positions(states)
    plan = [st if st[0] == "descend" else (st[0], st[1], batch) for st in PLAN]
    games, log = run_trees(m, plan, seed=n + trees)
    assert m.status() == 0
    final_pv = m.trees_principal_variation(32)
    for t, g in enumerate(games):
        replay_solo(s, states[g:g + 1], t, g, log, f"{n}x{n} T={trees} warps={warps}")
        assert list(s.tree_principal_variation(32)) == list(final_pv[0][g, :final_pv[1][g]])
    assert s.status() == 0
    assert np.array_equal(counters_tuple(m), counters_tuple(s)), "tz_counters = sum of the solo runs"
    m.close()
    s.close()


def oracle_pv(tree):
    buf = (O.C.c_uint16 * 64)()
    k = O.lib().tk_node_principal_variation(tree.ptr, buf, 64)
    return list(buf[:k])


def test_many_trees_against_the_oracle():
    """Every tree of one handle against the oracle's sequential Node::simulate_batch, descend and PV."""
    n, trees, batch = 5, 5, 16
    envs = openings(n, trees, seed=11)
    m = capi.BatchedMCTS(n, HK, trees, tree_batch=trees * batch, arena_slots=1 << 17)
    m.set_positions(games_to_states(envs))
    oracle_trees = [O.Tree() for _ in range(trees)]
    for move_no in range(3):
        for it in range(6):
            m.trees_simulate_batch(0.0, batch)
            for env, tree in zip(envs, oracle_trees):
                tree.simulate_batch("synthetic", env, 0.0, batch)
            for g, tree in enumerate(oracle_trees):
                dev = snapshot(m, [g])[0]
                assert_same_tree(dev, oracle_snapshot(tree, m, dev[0]["arena_used"]), f"move {move_no} batch {it} tree {g}")
        pv, ln = m.trees_principal_variation(64)
        moves = np.zeros(trees, np.uint16)
        for g, tree in enumerate(oracle_trees):
            assert list(pv[g, :ln[g]]) == oracle_pv(tree)
            moves[g] = pv[g, 0]
        m.trees_descend(moves)
        for g, (env, tree) in enumerate(zip(envs, oracle_trees)):
            tree.descend(int(moves[g]))
            O.play(env, int(moves[g]))
    assert m.status() == 0
    m.close()


def oracle_snapshot(tree, m, arena_used):
    """The oracle tree in the layout of `snapshot` (the oracle has no arena: its use is taken from the device)."""
    node = tree.node
    st = np.zeros((), capi.ROOT_DTYPE)
    st["arena_used"] = arena_used
    st["eval_tag"], st["eval_bits"] = node.evaluation.tag, node.evaluation.u.ply
    st["visit_count"], st["n_children"] = node.visit_count, node.n_children
    st["std_dev_bits"] = np.float32(node.std_dev).view(np.uint32)
    ch = oracle_children(node)
    full = {k: np.zeros(m.move_stride, ch[k].dtype) for k in ch}
    for k in ch:
        full[k][:node.n_children] = ch[k]
    return st, full


def recording_agent(name, n, hk, sizes):
    """tz_agent_fn forwarding to an oracle C agent; appends every batch size it is called with to `sizes`."""
    fn = getattr(O.lib(), f"tk_agent_{name}")
    fn.argtypes = [C.c_void_p, C.c_int, C.POINTER(O.Game), C.POINTER(C.c_uint16), C.POINTER(C.c_int), C.c_int,
                   C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]
    fn.restype = None

    def cb(_ctx, batch, envs, actions, n_actions, stride, logits, values, variances):
        sizes.append(batch)
        st = np.ctypeslib.as_array(C.cast(envs, C.POINTER(C.c_uint8)), shape=(batch * 384,)).view(capi.STATE_DTYPE)
        games = (O.Game * batch)(*[state_to_game(st[i], n, hk) for i in range(batch)])
        fn(None, batch, games, actions, n_actions, stride, logits, values, variances)

    return capi.AGENT_FN(cb)


TINUE_EASY = ["a3", "c1", "c2", "c3", "b3", "c3-"]  # mcts.rs:345-376
TINUE_DEEPER = ["a3", "a1", "b1", "c1"]  # mcts.rs:378-411


@pytest.mark.parametrize("batch", [3, 8, 24])
def test_known_results_and_early_ends_do_not_disturb_other_trees(batch):
    """The reference's tinue positions (descents end in known results and void the later ones in flight; the roots get
    solved and then fill no leaf), a finished game (solved from the start), and ordinary positions, in one call, with the
    reference's Simple agent.  The agent's batch is exactly the sum of what each tree queues alone."""
    n, hk = 3, 0
    finished = random_playout_states(n, hk, 5)[-1]
    assert O.terminal(finished) != O.T_NONE
    envs = [O.from_ptn_moves(n, hk, TINUE_EASY), O.new_opening(n, hk, 1, 0), finished,
            O.from_ptn_moves(n, hk, TINUE_DEEPER), O.new_opening(n, hk, 6, 1), O.from_ptn_moves(n, hk, TINUE_EASY)]
    states = games_to_states(envs)
    T, batches = len(envs), 80
    multi_sizes, solo_sizes = [], []
    m = capi.BatchedMCTS(n, hk, T, tree_batch=T * batch, arena_slots=1 << 18)
    m.set_agent(capi.AGENT_HOST, recording_agent("simple", n, hk, multi_sizes))
    m.set_positions(states)
    per_batch = []
    for _ in range(batches):
        before = len(multi_sizes)
        m.trees_simulate_batch(1.0, batch)
        per_batch.append(sum(multi_sizes[before:]))
    snaps = snapshot(m, range(T))
    assert m.status() == 0
    s = capi.BatchedMCTS(n, hk, 1, tree_batch=batch, arena_slots=1 << 18)
    s.set_agent(capi.AGENT_HOST, recording_agent("simple", n, hk, solo_sizes))
    want = np.zeros(batches, np.int64)
    for t in range(T):
        s.set_positions(states[t:t + 1])
        for i in range(batches):
            before = len(solo_sizes)
            s.tree_simulate_batch(1.0, batch)
            want[i] += sum(solo_sizes[before:])
        assert_same_tree(snaps[t], snapshot(s, [0])[0], f"tree {t}")
    assert s.status() == 0
    assert list(want) == per_batch, "queue total = sum of the per-tree counts"
    assert np.array_equal(counters_tuple(m), counters_tuple(s))
    stats = m.root_stats()
    assert stats["eval_tag"][2] != capi.E_VALUE, "the finished game's root is solved and fills no leaf"
    c = m.counters()
    assert c.known > 0 and c.known + c.evaluations == c.simulations
    m.close()
    s.close()


@pytest.mark.parametrize("n,trees", [(5, 3), (5, 6), (6, 2), (6, 4)])
def test_device_network_many_trees_equal_solo_trees(n, trees):
    """fp16 fused network with full-size weights.  128 leaves per tree: the solo handle runs the packed local chain
    (5 / 3 positions per CTA tile); 5x5 with 6 trees and 6x6 with 4 trees queue more positions than the packed layout
    takes (740 / 444), so their leaves run as dense rows, and must still give bit-identical trees."""
    batch, batches = 128, 4
    w = weights.random_init(n, seed=123)
    states = games_to_states(openings(n, trees, seed=3 * n))
    m = capi.BatchedMCTS(n, HK, trees, tree_batch=trees * batch, arena_slots=1 << 18)
    s = capi.BatchedMCTS(n, HK, 1, tree_batch=batch, arena_slots=1 << 18)
    for h in (m, s):
        network.set_weights(h, w, network.DTYPE_F16)
        h.set_agent(capi.AGENT_NETWORK)
    m.set_positions(states)
    games, log = run_trees(m, [("sim", 0.0, batch)] * batches + [("descend",), ("sim", 0.0, batch)], seed=n)
    assert m.status() == 0
    for t, g in enumerate(games):
        replay_solo(s, states[g:g + 1], t, g, log, f"{n}x{n} network T={trees}")
    assert s.status() == 0
    assert np.array_equal(counters_tuple(m), counters_tuple(s))
    m.close()
    s.close()


def test_masks_select_games_and_leave_the_others_alone():
    n, G, batch = 4, 6, 16
    mask = np.array([0, 1, 0, 0, 1, 0], np.uint8)
    states = games_to_states(openings(n, G, seed=21))
    m = capi.BatchedMCTS(n, HK, G, tree_batch=G * batch, arena_slots=1 << 16)
    m.set_positions(states)
    m.trees_simulate_batch(0.0, batch)  # every game: the unselected ones have trees worth keeping
    before_pos, before = m.positions(), snapshot(m, range(G))
    games, log = run_trees(m, [("sim", 0.0, batch)] * 3 + [("descend",), ("sim", 0.0, batch)], mask=mask)
    assert games == [1, 4]
    after_pos, after = m.positions(), snapshot(m, range(G))
    for g in range(G):
        if mask[g]:
            assert after_pos[g]["ply"] == before_pos[g]["ply"] + 1, "descend moves the selected games"
        else:
            assert after_pos[g].tobytes() == before_pos[g].tobytes(), f"game {g} position"
            assert_same_tree(after[g], before[g], f"unselected game {g}")
    pv, ln = m.trees_principal_variation(8, mask)
    assert all(ln[g] == 0 for g in range(G) if not mask[g]) and all(ln[g] >= 1 for g in games)
    # the selected trees are what they would be alone (game 0 of another handle, after the same first batch)
    s = capi.BatchedMCTS(n, HK, 1, tree_batch=batch, arena_slots=1 << 16)
    for t, g in enumerate(games):
        s.set_positions(states[g:g + 1])
        s.tree_simulate_batch(0.0, batch)
        replay_solo_from_here(s, t, g, log)
    assert m.status() == 0 and s.status() == 0
    m.close()
    s.close()


def replay_solo_from_here(s, t, g, log):
    for i, (step, moves, pv, snaps) in enumerate(log):
        if step[0] == "sim":
            s.tree_simulate_batch(step[1], step[2])
        else:
            s.tree_descend(int(moves[g]))
        assert_same_tree(snaps[t], snapshot(s, [0])[0], f"masked tree {t} step {i}")


def test_bad_arguments_change_nothing_and_an_empty_mask_is_a_no_op():
    n, G, batch = 4, 4, 16
    m = capi.BatchedMCTS(n, HK, G, tree_batch=2 * batch, arena_slots=1 << 16)
    m.set_positions(games_to_states(openings(n, G, seed=5)))
    m.trees_simulate_batch(0.0, 8)
    pos, snap, ctr = m.positions(), snapshot(m, range(G)), counters_tuple(m)

    def unchanged():
        assert m.positions().tobytes() == pos.tobytes()
        for g, (a, b) in enumerate(zip(snapshot(m, range(G)), snap)):
            assert_same_tree(a, b, f"game {g}")
        assert np.array_equal(counters_tuple(m), ctr)

    with pytest.raises(capi.TakzeroError):
        m.trees_simulate_batch(0.0, 0)
    with pytest.raises(capi.TakzeroError, match="tree_batch"):
        m.trees_simulate_batch(0.0, batch)  # 4 games x 16 > 32
    with pytest.raises(capi.TakzeroError, match="tree_batch"):
        m.trees_simulate_batch(0.0, 11, np.array([1, 1, 1, 0], np.uint8))
    with pytest.raises(capi.TakzeroError):
        m.trees_principal_variation(0)
    none = np.zeros(G, np.uint8)
    m.trees_simulate_batch(0.0, batch, none)
    m.trees_descend(np.zeros(G, np.uint16), none)
    pv, ln = m.trees_principal_variation(8, none)
    assert not ln.any()
    launches = m.launch_count()
    unchanged()
    assert m.status() == 0
    m.trees_simulate_batch(0.0, 16, np.array([1, 0, 1, 0], np.uint8))  # 2 x 16 = tree_batch: allowed
    assert m.launch_count() > launches and m.status() == 0
    m.close()


def test_trees_calls_make_pending_selfplay_records_stale():
    """Records pending at a tz_trees_* call describe roots the call changed: they are dropped, as after tz_tree_*, so
    no finished game emits a target from before the call.  Without the call the same run emits such targets."""
    n, G, seed = 3, 16, 9
    sp = capi.SelfplayParams(4, 24, 0.0, 2, 32, 0.5, 9.0, 0.25, seed)
    first_plies = {}
    for call in (False, True):
        m = capi.BatchedMCTS(n, 0, G, arena_slots=1 << 14)
        m.new_openings(seed=seed)
        m.selfplay_record(True)
        m.selfplay_move(sp)
        m.selfplay_move(sp)
        plies = m.positions()["ply"].copy()
        if call:
            m.trees_simulate_batch(0.0, 1, np.eye(G, dtype=np.uint8)[0])
        targets, seen = [], set()  # the targets of every game's first finished game
        for _ in range(30):
            m.selfplay_move(sp)
            d = m.selfplay_read()
            new = [(int(d["target_game"][i]), int(d["target_env"][i]["ply"])) for i in range(d["n_targets"])]
            targets += [(g, p) for g, p in new if g not in seen]
            seen |= {g for g, _ in new}
        assert m.status() == 0 and targets
        first_plies[call] = [(g, p) for g, p in targets if g != 0 and p < plies[g]]
        m.close()
    assert first_plies[False], "without the call, targets from the first two moves are emitted"
    assert not first_plies[True], "pending records were dropped"


def test_analysis_positions_prints_each_tree_as_a_solo_run(tmp_path):
    """`analysis --positions FILE --batches K`: per position, in file order, its TPS, the root display of the REPL and
    the PV, as a one-tree handle leaves them after K simulate_batch calls on that position."""
    import os
    import subprocess

    from takzero_b200 import build as tz_build
    from test_gpu_analysis_host import node_display

    tz_build.build()
    exe = os.path.join(os.path.dirname(capi.LIB_PATH), "bin", "analysis")
    n, batch, K = 5, 16, 4
    envs = openings(n, 6, seed=31)
    lines = [O.to_tps(g) for g in envs]
    f = tmp_path / "positions.txt"
    f.write_text("\n".join(lines) + "\n")
    out = subprocess.run([exe, "--board", str(n), "--half-komi", str(HK), "--batch-size", str(batch), "--arena-slots",
                          str(1 << 16), "--positions", str(f), "--batches", str(K)], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0, out.stderr
    want = ""
    s = capi.BatchedMCTS(n, HK, 1, tree_batch=batch, arena_slots=1 << 16)
    for text, g in zip(lines, envs):
        s.set_positions(games_to_states([g]))
        for _ in range(K):
            s.tree_simulate_batch(0.0, batch)
        pv = [O.move_str(int(mv)) for mv in s.tree_principal_variation(64)]
        want += f"tps: {text}\n" + node_display(s) + "pv:" + "".join(" " + mv for mv in pv) + "\n"
    assert s.status() == 0
    s.close()
    assert out.stdout == want
