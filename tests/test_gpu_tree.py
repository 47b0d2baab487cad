"""GPU parity of the single-tree path used by `tei` / `analysis`: Node::simulate_simple, simulate_batch
(many leaves of ONE tree per network batch, visit increments as the only virtual loss), descend (tree
reuse) and principal_variation (takzero/src/search/node/mcts.rs:235-328, node/mod.rs:40-102) -- bit-exact
against the oracle."""
import numpy as np
import pytest

from oracle import oracle as O
from takzero_b200 import capi

from helpers import assert_tree_equal, games_to_states, host_agent_from_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _device_matching_math():
    O.lib().tk_set_exact_math(1)
    yield
    O.lib().tk_set_exact_math(0)


def oracle_pv(tree):
    buf = (O.C.c_uint16 * 64)()
    k = O.lib().tk_node_principal_variation(tree.ptr, buf, 64)
    return list(buf[:k])


@pytest.mark.parametrize("n,half_komi,batch", [(4, 4, 16), (5, 4, 32), (6, 4, 64)])
def test_simulate_batch_descend_and_pv(n, half_komi, batch):
    env = O.new_opening(n, half_komi, 3, 1)
    m = capi.BatchedMCTS(n, half_komi, batch, arena_slots=1 << 17)
    m.set_positions(games_to_states([env] * batch))
    tree = O.Tree()
    rng = np.random.default_rng(n)
    for move_no in range(6):
        for it in range(12):
            m.tree_simulate_batch(0.0, batch)
            tree.simulate_batch("synthetic", env, 0.0, batch)
            if it in (0, 5):
                assert_tree_equal(m, tree, f"move {move_no} batch {it}")
        assert_tree_equal(m, tree, f"move {move_no}")
        pv = list(m.tree_principal_variation())
        assert pv == oracle_pv(tree) and len(pv) >= 1
        # tei: play the best move, keep the subtree (tei/src/main.rs:175-184)
        best = pv[0]  # the first PV move is select_best_action of the root
        assert best == O.lib().tk_node_select_best_action(tree.ptr)
        # every other move descends to a visited sibling instead, to exercise reuse of a smaller subtree
        if move_no % 2 == 1:
            tbl = m.root_children()
            visited = [int(tbl["moves"][0, i]) for i in range(tbl["n"][0]) if tbl["visits"][0, i] > 0]
            best = visited[int(rng.integers(len(visited)))]
        m.tree_descend(best)
        tree.descend(best)
        O.play(env, best)
        assert_tree_equal(m, tree, f"after descend {move_no}")
    m.close()


def test_simulate_simple_matches_oracle():
    """mcts.rs:235-266 with the reference's `Simple` agent injected; ends in a solved root (tinue position)."""
    env = O.from_ptn_moves(3, 0, ["a3", "a1", "b1", "c1"])
    m = capi.BatchedMCTS(3, 0, 2, arena_slots=1 << 17)
    m.set_positions(games_to_states([env, env]))
    m.set_agent(capi.AGENT_HOST, host_agent_from_oracle("simple", 3, 0))
    tree = O.Tree()
    for i in range(3000):
        m.tree_simulate_simple(0.0)
        tree.simulate_simple("simple", env, 0.0)
        if i % 500 == 0:
            assert_tree_equal(m, tree, f"sim {i}")
    assert_tree_equal(m, tree, "final")
    m.close()


TINUE_EASY = ["a3", "c1", "c2", "c3", "b3", "c3-"]  # mcts.rs:345-376
TINUE_DEEPER = ["a3", "a1", "b1", "c1"]  # mcts.rs:378-411


@pytest.mark.parametrize("batch,agent,moves", [(1, "synthetic", TINUE_EASY), (3, "simple", TINUE_EASY),
                                               (8, "simple", TINUE_EASY), (40, "simple", TINUE_EASY),
                                               (16, "dummy", TINUE_EASY), (24, "simple", TINUE_DEEPER),
                                               (128, "simple", TINUE_DEEPER)])
def test_simulate_batch_with_known_results_in_flight(batch, agent, moves):
    """The 3x3 position of the reference's `find_tinue_easy` (mcts.rs:345-376), beta = 1, with the reference's test
    agents: within a few batches most descents end in known results.  Each of them is backed up at once and changes
    what every later descent of the same batch sees, the forward budget of 4 x batch gets used up before the batch is
    full, and the root ends up solved -- on the device the descents of a batch run as a speculative wavefront of
    several warps, so this is the case where later descents have to be taken back and started again.  Bit-exact against
    the sequential oracle after every batch."""
    env = O.from_ptn_moves(3, 0, moves)
    m = capi.BatchedMCTS(3, 0, 1, tree_batch=batch, arena_slots=1 << 20)  # one game = the tree; `batch` queue slots
    m.set_positions(games_to_states([env]))
    if agent != "synthetic":
        m.set_agent(capi.AGENT_HOST, host_agent_from_oracle(agent, 3, 0))
    tree = O.Tree()
    for it in range(120):
        m.tree_simulate_batch(1.0, batch)
        tree.simulate_batch(agent, env, 1.0, batch)
        assert_tree_equal(m, tree, f"batch {it}")
    assert m.status() == 0
    c = m.counters()
    assert c.known > 0 and c.known + c.evaluations == c.simulations
    if agent == "simple" and batch >= 8 and moves is TINUE_EASY:
        assert m.root_stats()[0]["eval_tag"] != 0, "the root of this position is solved well within 120 batches"
        assert c.known > c.evaluations, "most descents ended in known results"
    pv = list(m.tree_principal_variation())
    assert pv == oracle_pv(tree)
    m.close()


@pytest.mark.parametrize("n,half_komi,batch,batches", [(5, 4, 128, 40), (4, 4, 100, 60), (6, 4, 37, 60)])
@pytest.mark.parametrize("warps", [1, 2, 3, 5, 8])
def test_simulate_batch_is_sequential_whatever_the_wavefront(n, half_komi, batch, batches, warps):
    """Longer runs on one growing tree, with the descents / backups of a batch spread over 1..8 warps: a descent whose
    path ends early must not let later ones run ahead of the still longer descents before it (the ordering mistake
    this test was written for showed only with some warp counts).  Bit-exact after every batch."""
    env = O.new_opening(n, half_komi, 5, 0)
    m = capi.BatchedMCTS(n, half_komi, 1, tree_batch=batch, arena_slots=1 << 20)
    m.debug_tree_warps(warps)
    m.set_positions(games_to_states([env]))
    tree = O.Tree()
    for it in range(batches):
        m.tree_simulate_batch(0.25, batch)
        tree.simulate_batch("synthetic", env, 0.25, batch)
        assert_tree_equal(m, tree, f"batch {it}")
    assert m.status() == 0
    assert list(m.tree_principal_variation()) == oracle_pv(tree)
    m.close()


def test_simulate_batch_soak_with_tree_reuse():
    """tei's loop at its own batch size (128 leaves, tei/src/main.rs) for 300 batches on a 6x6 tree that is re-rooted
    every 60 batches (subtree kept): 38k descents through one growing tree, compared every 20 batches."""
    n, half_komi, batch = 6, 4, 128
    env = O.new_opening(n, half_komi, 2, 1)
    m = capi.BatchedMCTS(n, half_komi, 1, tree_batch=batch, arena_slots=1 << 22)
    m.set_positions(games_to_states([env]))
    tree = O.Tree()
    for it in range(300):
        m.tree_simulate_batch(0.0, batch)
        tree.simulate_batch("synthetic", env, 0.0, batch)
        if it % 20 == 19:
            assert_tree_equal(m, tree, f"batch {it}")
        if it % 60 == 59:
            best = int(m.tree_principal_variation()[0])
            assert best == O.lib().tk_node_select_best_action(tree.ptr)
            m.tree_descend(best)
            tree.descend(best)
            O.play(env, best)
            assert_tree_equal(m, tree, f"after descend at batch {it}")
    assert m.status() == 0
    m.close()
