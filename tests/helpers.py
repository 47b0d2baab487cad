"""Shared helpers of the parity tests: oracle <-> C-ABI state conversion, seeded playouts."""
from __future__ import annotations

import ctypes as C

import numpy as np

from oracle import oracle as O
from takzero_b200 import capi


def game_to_state(g: O.Game) -> np.ndarray:
    s = np.zeros((), dtype=capi.STATE_DTYPE)
    s["stack"] = np.frombuffer(g.stack, dtype=np.uint64)
    s["height"] = np.frombuffer(g.height, dtype=np.uint8)
    s["top"] = np.frombuffer(g.top, dtype=np.uint8)
    s["to_move"] = g.to_move
    s["stones"] = [g.stones[0], g.stones[1]]
    s["caps"] = [g.caps[0], g.caps[1]]
    s["ply"] = g.ply
    s["reversible_plies"] = g.reversible_plies
    return s


def games_to_states(games) -> np.ndarray:
    out = np.zeros(len(games), dtype=capi.STATE_DTYPE)
    for i, g in enumerate(games):
        out[i] = game_to_state(g)
    return out


def state_to_game(s, n: int, half_komi: int, rev_limit: int = 100) -> O.Game:
    g = O.new_game(n, half_komi)
    for i in range(capi.MAX_SQ):
        g.stack[i] = int(s["stack"][i])
        g.height[i] = int(s["height"][i])
        g.top[i] = int(s["top"][i])
    g.to_move = int(s["to_move"])
    g.stones[0], g.stones[1] = int(s["stones"][0]), int(s["stones"][1])
    g.caps[0], g.caps[1] = int(s["caps"][0]), int(s["caps"][1])
    g.ply = int(s["ply"])
    g.reversible_plies = int(s["reversible_plies"])
    g.reversible_limit = rev_limit
    return g


def states_equal(a, b) -> bool:
    """Equality on the meaningful bytes (stack bits above `height` and `top` of empty squares excluded)."""
    for f in ("height", "to_move", "stones", "caps", "ply", "reversible_plies"):
        if not np.array_equal(a[f], b[f]):
            return False
    h = a["height"].astype(np.int64)
    mask = np.where(h >= 64, np.uint64(0xFFFFFFFFFFFFFFFF), (np.uint64(1) << h.astype(np.uint64)) - np.uint64(1))
    if not np.array_equal(a["stack"] & mask, b["stack"] & mask):
        return False
    occupied = h > 0
    return np.array_equal(a["top"][occupied], b["top"][occupied])


def states_equal_bulk(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Vectorised `states_equal` over arrays of STATE_DTYPE: bool per record."""
    ok = np.ones(len(a), dtype=bool)
    for f in ("to_move", "ply", "reversible_plies"):
        ok &= a[f] == b[f]
    for f in ("height", "stones", "caps"):
        ok &= (a[f] == b[f]).all(axis=1)
    h = a["height"].astype(np.uint64)
    mask = np.where(h >= 64, np.uint64(0xFFFFFFFFFFFFFFFF), (np.uint64(1) << np.minimum(h, np.uint64(63))) - np.uint64(1))
    ok &= ((a["stack"] & mask) == (b["stack"] & mask)).all(axis=1)
    occupied = a["height"] > 0
    ok &= ((a["top"] == b["top"]) | ~occupied).all(axis=1)
    return ok


def random_playout_states(n: int, half_komi: int, seed: int, max_plies: int = 400, keep_terminal: bool = True):
    """Uniform random legal playout from a random opening; returns the list of oracle Games visited."""
    rng = np.random.default_rng(seed)
    g = O.new_opening(n, half_komi, int(rng.integers(8)), int(rng.integers(2)))
    out = [g.copy()]
    for _ in range(max_plies):
        if O.terminal(g) != O.T_NONE:
            break
        moves = O.possible_moves(g)
        O.play(g, moves[int(rng.integers(len(moves)))])
        if O.terminal(g) == O.T_NONE or keep_terminal:
            out.append(g.copy())
    return out


def oracle_children(node) -> dict:
    n = node.n_children
    d = {
        "moves": np.array([node.actions[i] for i in range(n)], dtype=np.uint16),
        "visits": np.array([node.children[i].visit_count for i in range(n)], dtype=np.uint32),
        "eval_tag": np.array([node.children[i].evaluation.tag for i in range(n)], dtype=np.uint32),
        "eval_bits": np.array([node.children[i].evaluation.u.ply for i in range(n)], dtype=np.uint32),
        "logit": np.array([node.children[i].logit for i in range(n)], dtype=np.float32),
        "prob": np.array([node.children[i].probability for i in range(n)], dtype=np.float32),
        "std_dev": np.array([node.children[i].std_dev for i in range(n)], dtype=np.float32),
    }
    return d


def assert_roots_equal(mcts: "capi.BatchedMCTS", ob: "O.Batched", what: str = ""):
    """Bit-exact comparison of every root and its children between the CUDA trees and the oracle's."""
    tbl = mcts.root_children()
    stats = mcts.root_stats()
    for g in range(mcts.G):
        node = ob.node(g)
        assert stats["n_children"][g] == node.n_children, f"{what} game {g}: child count"
        assert stats["visit_count"][g] == node.visit_count, f"{what} game {g}: root visits"
        assert stats["eval_tag"][g] == node.evaluation.tag, f"{what} game {g}: root eval tag"
        assert stats["eval_bits"][g] == node.evaluation.u.ply, f"{what} game {g}: root eval bits"
        assert stats["std_dev_bits"][g] == np.float32(node.std_dev).view(np.uint32), f"{what} game {g}: root std"
        oc = oracle_children(node)
        n = node.n_children
        for key in ("moves", "visits", "eval_tag", "eval_bits"):
            assert np.array_equal(tbl[key][g, :n], oc[key]), f"{what} game {g}: children {key}"
        for key in ("logit", "prob", "std_dev"):
            assert np.array_equal(tbl[key][g, :n].view(np.uint32), oc[key].view(np.uint32)), \
                f"{what} game {g}: children {key} bits"


def assert_tree_equal(m, tree, what):
    node = tree.node
    st = m.root_stats()[0]
    tbl = m.root_children()
    assert st["n_children"] == node.n_children, what
    assert st["visit_count"] == node.visit_count, what
    assert (st["eval_tag"], st["eval_bits"]) == (node.evaluation.tag, node.evaluation.u.ply), what
    oc = oracle_children(node)
    n = node.n_children
    for key in ("moves", "visits", "eval_tag", "eval_bits"):
        assert np.array_equal(tbl[key][0, :n], oc[key]), f"{what}: {key}"
    for key in ("logit", "prob", "std_dev"):
        assert np.array_equal(tbl[key][0, :n].view(np.uint32), oc[key].view(np.uint32)), f"{what}: {key}"


def host_agent_from_oracle(name: str, n: int, half_komi: int):
    """tz_agent_fn that forwards to one of the oracle's C agents ('dummy', 'simple', 'synthetic')."""
    fn = getattr(O.lib(), f"tk_agent_{name}")
    fn.argtypes = [C.c_void_p, C.c_int, C.POINTER(O.Game), C.POINTER(C.c_uint16), C.POINTER(C.c_int), C.c_int,
                   C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]
    fn.restype = None

    def cb(_ctx, batch, envs, actions, n_actions, stride, logits, values, variances):
        st = np.ctypeslib.as_array(C.cast(envs, C.POINTER(C.c_uint8)), shape=(batch * 384,)).view(capi.STATE_DTYPE)
        games = (O.Game * batch)(*[state_to_game(st[i], n, half_komi) for i in range(batch)])
        fn(None, batch, games, actions, n_actions, stride, logits, values, variances)

    return capi.AGENT_FN(cb)


FILTERS = 256


def to_bf16_bits(x: np.ndarray) -> np.ndarray:
    u = x.astype(np.float32).view(np.uint32)
    return ((u + np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1))) >> np.uint32(16)).astype(np.uint16)


def folded_layer(w, bn, conv_bias, cin_pad, f16):
    """The host restatement: conv [cout][cin][3][3] (+ BN, eval mode, eps 1e-5) -> the 16-bit blocks
    [cin_pad/64][9 taps, centre first][2 halves][8 k-chunks][128 n][8] and 256 f32 biases."""
    cout, cin = w.shape[:2]
    one, eps = np.float32(1.0), np.float32(1e-5)
    scale = np.ones(cout, np.float32)
    bias = np.zeros(FILTERS, np.float32)
    if bn is not None:
        bw, bb, bm, bv = bn
        scale = (bw * (one / np.sqrt(bv + eps, dtype=np.float32))).astype(np.float32)
        bias[:cout] = bb - bm * scale
    if conv_bias is not None:
        bias[:cout] = bias[:cout] + conv_bias * scale
    full = np.zeros((FILTERS, cin_pad, 9), np.float32)
    full[:cout, :cin] = (w.reshape(cout, cin, 9) * scale[:, None, None]).astype(np.float32)
    taps = [4, 0, 1, 2, 3, 5, 6, 7, 8]
    blk = full[:, :, taps]                                  # [co][ci][ti]
    blk = blk.reshape(2, 128, cin_pad // 64, 8, 8, 9)        # [half][nrow][kb][kc][e][ti]
    blk = blk.transpose(2, 5, 0, 3, 1, 4)                    # [kb][ti][half][kc][nrow][e]
    flat = np.ascontiguousarray(blk).reshape(-1)
    bits = flat.astype(np.float16).view(np.uint16) if f16 else to_bf16_bits(flat)
    return bits, bias
