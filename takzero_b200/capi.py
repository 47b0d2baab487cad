"""ctypes binding of libtakzero_b200.so (include/takzero_b200.h) and a thin host-side mirror of
the reference's `BatchedMCTS` (takzero/src/search/node/batched.rs:24-409).

This is host plumbing only: every call goes to the CUDA library; there is no Python or CPU
implementation of the search here, and loading fails loudly when the library is missing."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TZ_LIB") or os.path.join(_HERE, "libtakzero_b200.so")

MAX_SQ = 36
MAX_MOVES = 1024
MAX_PLIES = 1024

AGENT_SYNTHETIC, AGENT_HOST, AGENT_NETWORK = 0, 1, 2
T_NONE, T_WIN, T_LOSS, T_DRAW = 0, 1, 2, 3
E_VALUE, E_WIN, E_LOSS, E_DRAW = 0, 1, 2, 3


class State(C.Structure):
    """tz_state_t: fast-tak `Game` fields (384 bytes)."""

    _fields_ = [
        ("stack", C.c_uint64 * MAX_SQ),
        ("height", C.c_uint8 * MAX_SQ),
        ("top", C.c_uint8 * MAX_SQ),
        ("to_move", C.c_uint8),
        ("stones", C.c_uint8 * 2),
        ("caps", C.c_uint8 * 2),
        ("pad0", C.c_uint8),
        ("ply", C.c_uint16),
        ("reversible_plies", C.c_uint16),
        ("pad1", C.c_uint8 * 14),
    ]


assert C.sizeof(State) == 384

STATE_DTYPE = np.dtype(
    [
        ("stack", "<u8", (MAX_SQ,)),
        ("height", "u1", (MAX_SQ,)),
        ("top", "u1", (MAX_SQ,)),
        ("to_move", "u1"),
        ("stones", "u1", (2,)),
        ("caps", "u1", (2,)),
        ("pad0", "u1"),
        ("ply", "<u2"),
        ("reversible_plies", "<u2"),
        ("pad1", "u1", (14,)),
    ]
)
assert STATE_DTYPE.itemsize == 384


class Config(C.Structure):
    _fields_ = [
        ("board_n", C.c_int),
        ("half_komi", C.c_int),
        ("n_games", C.c_int),
        ("device", C.c_int),
        ("game_base", C.c_int),
        ("reversible_limit", C.c_int),
        ("move_stride", C.c_int),
        ("arena_slots", C.c_uint32),
        ("tree_batch", C.c_int),
    ]


class Counters(C.Structure):
    _fields_ = [("simulations", C.c_uint64), ("evaluations", C.c_uint64), ("known", C.c_uint64),
                ("expansions", C.c_uint64)]


class SelfplayParams(C.Structure):
    """tz_selfplay_t: the compile-time constants of selfplay/src/main.rs:36-52 as runtime fields."""

    _fields_ = [("sampled_actions", C.c_int), ("search_budget", C.c_uint32), ("beta", C.c_float),
                ("weighted_random_plies", C.c_int), ("sample_threshold", C.c_uint32),
                ("allowed_eval_drop", C.c_float), ("target_visitations", C.c_float), ("target_beta", C.c_float),
                ("seed", C.c_uint64)]


class ReanalyzeParams(C.Structure):
    """tz_reanalyze_t: SAMPLED_ACTIONS, SEARCH_BUDGET, UBE_TARGET_BETA of reanalyze/src/main.rs as runtime fields."""

    _fields_ = [("sampled_actions", C.c_int), ("search_budget", C.c_uint32), ("target_beta", C.c_float),
                ("seed", C.c_uint64)]


class SelfplayData(C.Structure):
    """tz_selfplay_data_t: caller buffers of tz_selfplay_read."""

    _fields_ = [("target_cap", C.c_size_t), ("policy_cap", C.c_size_t), ("replay_cap", C.c_size_t),
                ("move_cap", C.c_size_t),
                ("target_env", C.c_void_p), ("target_value", C.c_void_p), ("target_ube", C.c_void_p),
                ("target_n", C.c_void_p), ("target_offset", C.c_void_p), ("target_game", C.c_void_p),
                ("policy_moves", C.c_void_p), ("policy_probs", C.c_void_p),
                ("replay_start", C.c_void_p), ("replay_result", C.c_void_p), ("replay_terminal", C.c_void_p),
                ("replay_length", C.c_void_p), ("replay_offset", C.c_void_p), ("replay_game", C.c_void_p),
                ("replay_exploration", C.c_void_p), ("replay_moves", C.c_void_p),
                ("n_targets", C.c_size_t), ("n_policy", C.c_size_t), ("n_replays", C.c_size_t),
                ("n_moves", C.c_size_t), ("high_water_bytes", C.c_size_t)]


# tz_selfplay_data_t arrays: name -> (count field, dtype)
SELFPLAY_FIELDS = {
    "target_env": ("n_targets", STATE_DTYPE), "target_value": ("n_targets", np.float32),
    "target_ube": ("n_targets", np.float32), "target_n": ("n_targets", np.int32),
    "target_offset": ("n_targets", np.uint64), "target_game": ("n_targets", np.int32),
    "policy_moves": ("n_policy", np.uint16), "policy_probs": ("n_policy", np.float32),
    "replay_start": ("n_replays", STATE_DTYPE), "replay_result": ("n_replays", np.int32),
    "replay_terminal": ("n_replays", np.int32), "replay_length": ("n_replays", np.int32),
    "replay_offset": ("n_replays", np.uint64), "replay_game": ("n_replays", np.int32),
    "replay_exploration": ("n_replays", np.uint8), "replay_moves": ("n_moves", np.uint16),
}
STATUS_TARGETS_FULL = 1024


class Profile(C.Structure):
    _fields_ = [("ms", C.c_double * 8), ("launches", C.c_uint64 * 8), ("locksteps", C.c_uint64),
                ("positions", C.c_uint64)]


PROFILE_CATEGORIES = ("select", "encode", "conv_input", "conv_tower", "conv_policy", "heads_gather", "expand",
                      "agent_synthetic")

ROOT_DTYPE = np.dtype([("eval_tag", "<u4"), ("eval_bits", "<u4"), ("visit_count", "<u4"),
                       ("std_dev_bits", "<u4"), ("n_children", "<u4"), ("arena_used", "<u4")])

AGENT_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(State), C.POINTER(C.c_uint16), C.POINTER(C.c_int),
                       C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float))


class TakzeroError(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m takzero_b200.build` "
            "(takzero_b200 has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    P, vp, i32, u32, u64, f32 = C.POINTER, C.c_void_p, C.c_int, C.c_uint32, C.c_uint64, C.c_float
    sig = {
        "tz_last_error": ([], C.c_char_p),
        "tz_version": ([], C.c_char_p),
        "tz_create": ([P(Config), P(vp)], i32),
        "tz_destroy": ([vp], None),
        "tz_sync": ([vp], i32),
        "tz_status": ([vp, P(u32)], i32),
        "tz_clear_status": ([vp], i32),
        "tz_info": ([vp, P(i32), P(u32), P(i32), P(i32)], i32),
        "tz_host_alloc": ([C.c_size_t], vp),
        "tz_host_free": ([vp], None),
        "tz_legal_moves": ([vp, vp, i32, i32, vp, vp], i32),
        "tz_apply": ([vp, vp, vp, i32, vp], i32),
        "tz_result": ([vp, vp, i32, vp], i32),
        "tz_game_result": ([vp, vp, i32, vp], i32),
        "tz_set_positions": ([vp, vp, vp], i32),
        "tz_get_positions": ([vp, vp], i32),
        "tz_new_openings": ([vp, vp, vp, vp, u64], i32),
        "tz_reset_roots": ([vp, vp], i32),
        "tz_random_steps": ([vp, vp, i32, u64], i32),
        "tz_set_agent": ([vp, i32, vp, vp], i32),
        "tz_simulate": ([vp, vp], i32),
        "tz_gumbel_sequential_halving": ([vp, vp, i32, u32, vp, i32, u64, vp], i32),
        "tz_last_gumbel": ([vp, vp, i32], i32),
        "tz_step": ([vp, vp], i32),
        "tz_restart_terminal": ([vp, vp, vp, u64, vp], i32),
        "tz_finished_replay": ([vp, i32, vp, vp, i32], i32),
        "tz_replay": ([vp, i32, vp, vp, i32], i32),
        "tz_root_children": ([vp, i32, vp, vp, vp, vp, vp, vp, vp, vp], i32),
        "tz_root_stats": ([vp, vp], i32),
        "tz_targets": ([vp, f32, f32, i32, vp, vp, vp, vp], i32),
        "tz_select_best": ([vp, vp], i32),
        "tz_select_selfplay": ([vp, i32, u32, f32, vp, u64, vp], i32),
        "tz_counters": ([vp, P(Counters)], i32),
        "tz_set_root_priors": ([vp, i32, vp, vp], i32),
        "tz_tree_simulate_simple": ([vp, f32], i32),
        "tz_tree_simulate_batch": ([vp, f32, i32], i32),
        "tz_debug_tree_warps": ([vp, i32], i32),
        "tz_tree_descend": ([vp, C.c_uint16], i32),
        "tz_tree_principal_variation": ([vp, vp, i32], i32),
        "tz_trees_simulate_batch": ([vp, vp, f32, i32], i32),
        "tz_trees_descend": ([vp, vp, vp], i32),
        "tz_trees_principal_variation": ([vp, vp, i32, vp, vp], i32),
        "tz_selfplay_move": ([vp, P(SelfplayParams)], i32),
        "tz_launch_count": ([vp, P(u64)], i32),
        "tz_selfplay_record": ([vp, i32, C.c_size_t, C.c_size_t], i32),
        "tz_selfplay_read": ([vp, P(SelfplayData)], i32),
        "tz_stage_positions": ([vp, vp, C.c_size_t], i32),
        "tz_reanalyze_batch": ([vp, vp, P(ReanalyzeParams)], i32),
        "tz_reanalyze_read": ([vp, i32, vp, vp, vp, vp, vp], i32),
        "tz_profile_begin": ([vp, i32], i32),
        "tz_profile_end": ([vp, P(Profile)], i32),
        "tz_timer_start": ([vp], i32),
        "tz_timer_stop": ([vp, P(C.c_double)], i32),
    }
    for name, (args, res) in sig.items():
        fn = getattr(L, name)
        fn.argtypes = args
        fn.restype = res
    L._optional = {}
    _lib = L
    return L


def declare(name, args, res):
    """Declare a further export (used by modules that add entry points, e.g. the network)."""
    fn = getattr(lib(), name)
    fn.argtypes = args
    fn.restype = res
    return fn


def pinned_array(shape, dtype) -> np.ndarray:
    """numpy view of pinned host memory from tz_host_alloc (kept alive by the returned array's base)."""
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    p = lib().tz_host_alloc(max(nbytes, 1))
    if not p:
        raise MemoryError("tz_host_alloc failed")
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(p)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    return arr


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _check(rc: int):
    if rc < 0:
        raise TakzeroError(f"{lib().tz_last_error().decode()} (code {rc})")
    return rc


def _arr(x, dtype, shape=None) -> np.ndarray:
    a = np.ascontiguousarray(x, dtype=dtype)
    if shape is not None and a.shape != shape:
        raise ValueError(f"expected shape {shape}, got {a.shape}")
    return a


class BatchedMCTS:
    """Host mirror of `BatchedMCTS<BATCH_SIZE, Env>`; all state lives on the device."""

    def __init__(self, board_n: int, half_komi: int, n_games: int, device: int = 0, game_base: int = 0,
                 reversible_limit: int = 0, move_stride: int = 0, arena_slots: int = 0, tree_batch: int = 0):
        self._h = C.c_void_p()
        cfg = Config(board_n, half_komi, n_games, device, game_base, reversible_limit, move_stride, arena_slots,
                     tree_batch)
        _check(lib().tz_create(C.byref(cfg), C.byref(self._h)))
        self.n = board_n
        self.half_komi = half_komi
        self.G = n_games
        self.game_base = game_base
        ms, slots, ic, oc = C.c_int(), C.c_uint32(), C.c_int(), C.c_int()
        _check(lib().tz_info(self._h, C.byref(ms), C.byref(slots), C.byref(ic), C.byref(oc)))
        self.move_stride, self.arena_slots = ms.value, slots.value
        self.input_channels, self.output_channels = ic.value, oc.value
        self._agent_cb = None

    @property
    def handle(self):
        return self._h

    def close(self):
        if getattr(self, "_h", None):
            lib().tz_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- rules hooks -----------------------------------------------------------------
    def legal_moves(self, states: np.ndarray, stride: Optional[int] = None):
        states = _arr(states, STATE_DTYPE)
        stride = stride or self.move_stride
        moves = np.zeros((len(states), stride), dtype=np.uint16)
        n = np.zeros(len(states), dtype=np.int32)
        _check(lib().tz_legal_moves(self._h, _ptr(states), len(states), stride, _ptr(moves), _ptr(n)))
        return moves, n

    def apply(self, states: np.ndarray, moves):
        states = _arr(states, STATE_DTYPE).copy()
        moves = _arr(moves, np.uint16, (len(states),))
        ok = np.zeros(len(states), dtype=np.int32)
        _check(lib().tz_apply(self._h, _ptr(states), _ptr(moves), len(states), _ptr(ok)))
        return states, ok

    def result(self, states: np.ndarray):
        states = _arr(states, STATE_DTYPE)
        out = np.zeros(len(states), dtype=np.int32)
        _check(lib().tz_result(self._h, _ptr(states), len(states), _ptr(out)))
        return out

    def game_result(self, states: np.ndarray):
        """0 ongoing, 1 R-0, 2 0-R, 3 F-0, 4 0-F, 5 draw."""
        states = _arr(states, STATE_DTYPE)
        out = np.zeros(len(states), dtype=np.int32)
        _check(lib().tz_game_result(self._h, _ptr(states), len(states), _ptr(out)))
        return out

    # ---- positions --------------------------------------------------------------------
    def set_positions(self, states: np.ndarray, mask=None):
        states = _arr(states, STATE_DTYPE, (self.G,))
        m = None if mask is None else _arr(mask, np.uint8, (self.G,))
        _check(lib().tz_set_positions(self._h, _ptr(states), _ptr(m)))

    def positions(self) -> np.ndarray:
        out = np.zeros(self.G, dtype=STATE_DTYPE)
        _check(lib().tz_get_positions(self._h, _ptr(out)))
        return out

    def new_openings(self, sym=None, adj=None, seed: int = 0, mask=None):
        s = None if sym is None else _arr(sym, np.int32, (self.G,))
        a = None if adj is None else _arr(adj, np.int32, (self.G,))
        m = None if mask is None else _arr(mask, np.uint8, (self.G,))
        _check(lib().tz_new_openings(self._h, _ptr(m), _ptr(s), _ptr(a), seed))

    def random_steps(self, steps: int, seed: int = 0, mask=None):
        """The random part of `new_opening_with_random_steps` (env.rs:81-96)."""
        m = None if mask is None else _arr(mask, np.uint8, (self.G,))
        _check(lib().tz_random_steps(self._h, _ptr(m), steps, seed))

    def reset_roots(self, mask=None):
        m = None if mask is None else _arr(mask, np.uint8, (self.G,))
        _check(lib().tz_reset_roots(self._h, _ptr(m)))

    # ---- search -----------------------------------------------------------------------
    def set_agent(self, kind: int, fn=None):
        cb = None
        if kind == AGENT_HOST:
            cb = fn if isinstance(fn, AGENT_FN) else AGENT_FN(fn)
        self._agent_cb = cb
        _check(lib().tz_set_agent(self._h, kind, C.cast(cb, C.c_void_p) if cb else None, None))

    def simulate(self, betas=None):
        b = None if betas is None else _arr(betas, np.float32, (self.G,))
        _check(lib().tz_simulate(self._h, _ptr(b)))

    def gumbel_sequential_halving(self, betas, sampled_actions: int, search_budget: int, gumbel=None,
                                  seed: int = 0) -> np.ndarray:
        b = None if betas is None else _arr(betas, np.float32, (self.G,))
        out = np.zeros(self.G, dtype=np.uint16)
        if gumbel is not None:
            gum = _arr(gumbel, np.float32)
            assert gum.ndim == 2 and gum.shape[0] == self.G
            _check(lib().tz_gumbel_sequential_halving(self._h, _ptr(b), sampled_actions, search_budget,
                                                      _ptr(gum), gum.shape[1], seed, _ptr(out)))
        else:
            _check(lib().tz_gumbel_sequential_halving(self._h, _ptr(b), sampled_actions, search_budget,
                                                      None, 0, seed, _ptr(out)))
        return out

    def last_gumbel(self) -> np.ndarray:
        out = np.zeros((self.G, self.move_stride), dtype=np.float32)
        _check(lib().tz_last_gumbel(self._h, _ptr(out), self.move_stride))
        return out

    def step(self, moves):
        m = _arr(moves, np.uint16, (self.G,))
        _check(lib().tz_step(self._h, _ptr(m)))

    def restart_terminal_envs(self, sym=None, adj=None, seed: int = 0) -> np.ndarray:
        s = None if sym is None else _arr(sym, np.int32, (self.G,))
        a = None if adj is None else _arr(adj, np.int32, (self.G,))
        out = np.zeros(self.G, dtype=np.int32)
        _check(lib().tz_restart_terminal(self._h, _ptr(s), _ptr(a), seed, _ptr(out)))
        return out

    def _replay(self, fn, game: int):
        start = np.zeros(1, dtype=STATE_DTYPE)
        moves = np.zeros(MAX_PLIES, dtype=np.uint16)
        n = _check(fn(self._h, game, _ptr(start), _ptr(moves), MAX_PLIES))
        return start[0], moves[:n].copy()

    def finished_replay(self, game: int):
        return self._replay(lib().tz_finished_replay, game)

    def replay(self, game: int):
        return self._replay(lib().tz_replay, game)

    # ---- read-backs ---------------------------------------------------------------------
    def root_children(self, stride: Optional[int] = None) -> dict:
        stride = stride or self.move_stride
        G = self.G
        out = {
            "n": np.zeros(G, dtype=np.int32),
            "moves": np.zeros((G, stride), dtype=np.uint16),
            "visits": np.zeros((G, stride), dtype=np.uint32),
            "eval_tag": np.zeros((G, stride), dtype=np.uint32),
            "eval_bits": np.zeros((G, stride), dtype=np.uint32),
            "logit": np.zeros((G, stride), dtype=np.float32),
            "prob": np.zeros((G, stride), dtype=np.float32),
            "std_dev": np.zeros((G, stride), dtype=np.float32),
        }
        _check(lib().tz_root_children(self._h, stride, _ptr(out["n"]), _ptr(out["moves"]), _ptr(out["visits"]),
                                      _ptr(out["eval_tag"]), _ptr(out["eval_bits"]), _ptr(out["logit"]),
                                      _ptr(out["prob"]), _ptr(out["std_dev"])))
        return out

    def root_stats(self) -> np.ndarray:
        out = np.zeros(self.G, dtype=ROOT_DTYPE)
        _check(lib().tz_root_stats(self._h, _ptr(out)))
        return out

    def targets(self, visitations: float, beta: float, stride: Optional[int] = None, with_moves: bool = False, out=None):
        """`out` = (policy, ube, n[, moves]) arrays to fill (e.g. pinned memory from pinned_array: the copies are then
        asynchronous DMA instead of staged through pageable memory)."""
        stride = stride or self.move_stride
        if out is not None:
            pol, ube, n = out[0], out[1], out[2]
            mv = out[3] if with_moves else None
        else:
            pol = np.zeros((self.G, stride), dtype=np.float32)
            ube = np.zeros(self.G, dtype=np.float32)
            n = np.zeros(self.G, dtype=np.int32)
            mv = np.zeros((self.G, stride), dtype=np.uint16) if with_moves else None
        _check(lib().tz_targets(self._h, visitations, beta, stride, _ptr(pol), _ptr(ube), _ptr(n), _ptr(mv)))
        return (pol, ube, n, mv) if with_moves else (pol, ube, n)

    def select_best_actions(self) -> np.ndarray:
        out = np.zeros(self.G, dtype=np.uint16)
        _check(lib().tz_select_best(self._h, _ptr(out)))
        return out

    def select_actions_in_selfplay(self, weighted_random_plies: int, threshold: int = 32, allowed_drop: float = 0.5,
                                   randoms=None, seed: int = 0) -> np.ndarray:
        r = None if randoms is None else _arr(randoms, np.uint64, (self.G,))
        out = np.zeros(self.G, dtype=np.uint16)
        _check(lib().tz_select_selfplay(self._h, weighted_random_plies, threshold, allowed_drop, _ptr(r), seed,
                                        _ptr(out)))
        return out

    def apply_noise(self, noise: np.ndarray, ratio: float) -> None:
        """BatchedMCTS::apply_noise with injected Dirichlet samples `noise` [G, move_stride] (the reference
        draws them from rand_distr, whose stream is not pinned): p' = p*(1-ratio) + noise*ratio, logit' = ln p'
        in f32 on the host (node/noise.rs:18-25), stored back into the roots."""
        tbl = self.root_children()
        noise = _arr(noise, np.float32, (self.G, self.move_stride))
        r = np.float32(ratio)
        prob = (tbl["prob"] * (np.float32(1.0) - r) + noise * r).astype(np.float32)
        with np.errstate(divide="ignore"):
            logit = np.log(prob, dtype=np.float32)
        _check(lib().tz_set_root_priors(self._h, self.move_stride, _ptr(prob), _ptr(logit)))

    def counters(self) -> Counters:
        c = Counters()
        _check(lib().tz_counters(self._h, C.byref(c)))
        return c

    # ---- single tree (game 0): the reference's Node::simulate_simple / simulate_batch / descend / PV ----
    def tree_simulate_simple(self, beta: float = 0.0) -> None:
        _check(lib().tz_tree_simulate_simple(self._h, beta))

    def tree_simulate_batch(self, beta: float, batch_size: int) -> None:
        _check(lib().tz_tree_simulate_batch(self._h, beta, batch_size))

    def debug_tree_warps(self, warps: int) -> None:
        """Test hook: warps of the single-tree wavefront kernels (0 = default 8); changes the interleaving only."""
        _check(lib().tz_debug_tree_warps(self._h, int(warps)))

    def tree_descend(self, move: int) -> None:
        _check(lib().tz_tree_descend(self._h, int(move)))

    def tree_principal_variation(self, cap: int = 64) -> np.ndarray:
        out = np.zeros(cap, dtype=np.uint16)
        n = _check(lib().tz_tree_principal_variation(self._h, _ptr(out), cap))
        return out[:n].copy()

    # ---- many single trees at once: the tree of every selected game (mask [G], None = every game) ----
    def trees_simulate_batch(self, beta: float, batch_size: int, mask=None) -> None:
        """Node::simulate_batch on every selected game's tree, one network batch for all of them
        (selected games * batch_size <= max(n_games, tree_batch))."""
        m = None if mask is None else _arr(mask, np.uint8, (self.G,))
        _check(lib().tz_trees_simulate_batch(self._h, _ptr(m), beta, batch_size))

    def trees_descend(self, moves, mask=None) -> None:
        """Node::descend + env.step of every selected game (moves [G]; unselected games' entries are ignored)."""
        mv = _arr(moves, np.uint16, (self.G,))
        m = None if mask is None else _arr(mask, np.uint8, (self.G,))
        _check(lib().tz_trees_descend(self._h, _ptr(m), _ptr(mv)))

    def trees_principal_variation(self, cap: int = 64, mask=None):
        """Per game: (moves [G][cap] uint16, lengths [G] int32); length 0 for unselected games."""
        m = None if mask is None else _arr(mask, np.uint8, (self.G,))
        out = np.zeros((self.G, cap), dtype=np.uint16)
        n = np.zeros(self.G, dtype=np.int32)
        _check(lib().tz_trees_principal_variation(self._h, _ptr(m), cap, _ptr(out), _ptr(n)))
        return out, n

    def selfplay_move(self, params: SelfplayParams) -> None:
        """One whole self-play move on the device, asynchronous (see tz_selfplay_move)."""
        _check(lib().tz_selfplay_move(self._h, C.byref(params)))

    def selfplay_record(self, enable: bool = True, bytes_per_game: int = 0, output_bytes: int = 0) -> None:
        """Keep the training data of selfplay_move on the device (0 = default sizes; see tz_selfplay_record)."""
        _check(lib().tz_selfplay_record(self._h, 1 if enable else 0, int(bytes_per_game), int(output_bytes)))

    def selfplay_read(self, capacity: Optional[dict] = None) -> dict:
        """Completed targets and finished replays since the last read, as numpy arrays (empties the queue).

        Targets come per finished game in ascending game order, each game's from its last ply to its first; target i
        has policy entries policy_moves / policy_probs[target_offset[i] : + target_n[i]], replay j its moves
        replay_moves[replay_offset[j] : + replay_length[j]].  `capacity` = {"n_targets": .., "n_policy": ..,
        "n_replays": .., "n_moves": ..} reads with fixed buffers (TakzeroError when too small); None sizes them from
        the queue.  Also returns "high_water_bytes"."""
        io = SelfplayData()
        if capacity is None:
            rc = lib().tz_selfplay_read(self._h, C.byref(io))  # capacities 0: reports the counts
            if rc == 0:
                return self._selfplay_arrays(io, {k: 0 for k in ("n_targets", "n_policy", "n_replays", "n_moves")})
            if rc != -1 or not (io.n_targets or io.n_policy or io.n_replays or io.n_moves):
                _check(rc)
            capacity = {k: getattr(io, k) for k in ("n_targets", "n_policy", "n_replays", "n_moves")}
        out = {name: np.zeros(capacity[cnt], dtype=dt) for name, (cnt, dt) in SELFPLAY_FIELDS.items()}
        io = SelfplayData()
        io.target_cap, io.policy_cap = capacity["n_targets"], capacity["n_policy"]
        io.replay_cap, io.move_cap = capacity["n_replays"], capacity["n_moves"]
        for name, a in out.items():
            setattr(io, name, a.ctypes.data_as(C.c_void_p).value if a.size else None)
        _check(lib().tz_selfplay_read(self._h, C.byref(io)))
        return self._selfplay_arrays(io, capacity, out)

    @staticmethod
    def _selfplay_arrays(io, capacity, out=None) -> dict:
        res = {}
        for name, (cnt, dt) in SELFPLAY_FIELDS.items():
            n = getattr(io, cnt)
            res[name] = out[name][:n].copy() if out is not None else np.zeros(0, dtype=dt)
        for k in ("n_targets", "n_policy", "n_replays", "n_moves", "high_water_bytes"):
            res[k] = int(getattr(io, k))
        return res

    # ---- reanalyze (reanalyze/src/main.rs:147-235) ---------------------------------------------------------
    def stage_positions(self, states: np.ndarray) -> None:
        """Upload the replay buffer's positions once; batches then pick their roots by index."""
        states = _arr(states, STATE_DTYPE)
        _check(lib().tz_stage_positions(self._h, _ptr(states), len(states)))

    def reanalyze_batch(self, pool_indices, params: ReanalyzeParams) -> None:
        """One batch on the device, asynchronous: fresh roots from the staged positions (None: the current ones),
        search, targets."""
        idx = None if pool_indices is None else _arr(pool_indices, np.uint32, (self.G,))
        _check(lib().tz_reanalyze_batch(self._h, _ptr(idx), C.byref(params)))

    def reanalyze_read(self, out=None) -> dict:
        """Targets of the last batch: improved policy, moves, child counts, UBE and value targets."""
        if out is None:
            out = {"policy": np.zeros((self.G, self.move_stride), np.float32),
                   "moves": np.zeros((self.G, self.move_stride), np.uint16),
                   "ube": np.zeros(self.G, np.float32), "value": np.zeros(self.G, np.float32),
                   "n": np.zeros(self.G, np.int32)}
        _check(lib().tz_reanalyze_read(self._h, self.move_stride, _ptr(out["policy"]), _ptr(out["ube"]),
                                       _ptr(out["value"]), _ptr(out["n"]), _ptr(out["moves"])))
        return out

    def launch_count(self) -> int:
        out = C.c_uint64()
        _check(lib().tz_launch_count(self._h, C.byref(out)))
        return out.value

    def profile_begin(self, sample_every: int) -> None:
        _check(lib().tz_profile_begin(self._h, sample_every))

    def profile_end(self) -> Profile:
        p = Profile()
        _check(lib().tz_profile_end(self._h, C.byref(p)))
        return p

    def timer_start(self) -> None:
        _check(lib().tz_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_double()
        _check(lib().tz_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def status(self) -> int:
        bits = C.c_uint32()
        _check(lib().tz_status(self._h, C.byref(bits)))
        return bits.value

    def sync(self):
        _check(lib().tz_sync(self._h))
