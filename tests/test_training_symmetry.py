"""The 8 board symmetries of training batches (tz_training_batch), restated in Python and checked against the oracle's
rules on 3x3 to 6x6.  tests/test_gpu_training_batch.py compares the device kernel with this restatement.

A symmetry t maps square (row, col) by, in this order: bit 0 mirrors the column, bit 1 mirrors the row, bit 2 swaps
row and column.  A spread keeps its pattern byte and maps its direction (0 '+', 1 '-', 2 '<', 3 '>') alike."""
import numpy as np
import pytest

from draws import rng_hash
from oracle import oracle as O

REVERSIBLE_LIMIT = 100


def sym_square(t: int, n: int, row: int, col: int):
    if t & 1:
        col = n - 1 - col
    if t & 2:
        row = n - 1 - row
    if t & 4:
        row, col = col, row
    return row, col


def sym_move(t: int, n: int, m: int) -> int:
    col, row, kd, pat = m & 7, (m >> 3) & 7, (m >> 6) & 3, m >> 8
    row, col = sym_square(t, n, row, col)
    if pat:
        if t & 1 and kd >= 2:
            kd ^= 1  # '<' <-> '>'
        if t & 2 and kd < 2:
            kd ^= 1  # '+' <-> '-'
        if t & 4:
            kd = 3 - kd  # '+' <-> '>', '-' <-> '<'
    return col | (row << 3) | (kd << 6) | (pat << 8)


def sym_state(t: int, n: int, rec: np.ndarray) -> np.ndarray:
    """One tz_state_t record (uint8 [384]) under symmetry t: squares moved, everything else kept."""
    rec = np.ascontiguousarray(rec).view(np.uint8).reshape(384)
    out = rec.copy()
    stack, height, top = rec[:288].view(np.uint64), rec[288:324], rec[324:360]
    o_stack, o_height, o_top = out[:288].view(np.uint64), out[288:324], out[324:360]
    for sq in range(n * n):
        r, c = sym_square(t, n, sq // n, sq % n)
        to = r * n + c
        o_stack[to], o_height[to], o_top[to] = stack[sq], height[sq], top[sq]
    return out


def draw_index(seed: int, i: int, size: int) -> int:
    return (rng_hash(seed, i, 0, 0) * size) >> 64


def draw_symmetry(seed: int, i: int) -> int:
    return rng_hash(seed, i, 1, 0) & 7


def output_channels(n: int) -> int:
    return 3 + 4 * ((1 << n) - 2)


def has_move_index(n: int, m: int) -> bool:
    """The host check of tz_target_buffer_append: move_index exists for m on an n x n board."""
    col, row, kd, pat = m & 7, (m >> 3) & 7, (m >> 6) & 3, m >> 8
    if row >= n or col >= n:
        return False
    if pat == 0:
        return kd <= 2
    if pat & ((1 << (8 - n)) - 1):
        return False
    return 1 <= pat >> (8 - n) <= (1 << n) - 2


def positions(n: int, seed: int, count: int):
    return O.playout_positions(n, 4, seed, 4, count, reversible_limit=REVERSIBLE_LIMIT)


@pytest.mark.parametrize("n", [3, 4, 5, 6])
def test_symmetries_commute_with_the_rules(oracle, n):
    pp = positions(n, 11 + n, 160)
    assert (pp["terminal"] != 0).any(), "the playouts include finished games"
    nn, oc = n * n, output_channels(n)
    for i in range(len(pp["states"])):
        legal = [int(m) for m in pp["moves"][i, :pp["n_moves"][i]]]
        assert all(has_move_index(n, m) for m in legal)
        for t in range(8):
            g = O.unpack_games(sym_state(t, n, pp["states"][i]), n, 4, REVERSIBLE_LIMIT)[0]
            mapped = [sym_move(t, n, m) for m in legal]
            assert sorted(mapped) == sorted(O.possible_moves(g)), (n, i, t)
            assert O.terminal(g) == pp["terminal"][i] and O.result(g) == O.result(pp["games"][i]), (n, i, t)
            idx = [O.move_index(n, m) for m in mapped]
            assert all(0 <= k < oc * nn for k in idx) and len(set(idx)) == len(idx), (n, i, t)
            assert all(has_move_index(n, m) for m in mapped)


@pytest.mark.parametrize("n", [3, 4, 5, 6])
def test_symmetries_form_the_dihedral_group(n):
    # every square with every direction, and the placements: the images determine a symmetry
    pat = 1 << 7
    probe = [col | (row << 3) | (kd << 6) | (p << 8) for row in range(n) for col in range(n) for kd in range(4)
             for p in (0, pat) if p or kd < 3]
    image = {t: tuple(sym_move(t, n, m) for m in probe) for t in range(8)}
    assert image[0] == tuple(probe), "symmetry 0 is the identity"
    assert len(set(image.values())) == 8, "the 8 symmetries are distinct"
    for t in range(8):
        assert sorted(image[t]) == sorted(probe), "a symmetry permutes the moves"
    for a in range(8):
        for b in range(8):
            composed = tuple(sym_move(b, n, sym_move(a, n, m)) for m in probe)
            assert composed in image.values(), f"{b} after {a} is not one of the 8"
        assert any(tuple(sym_move(b, n, sym_move(a, n, m)) for m in probe) == tuple(probe) for b in range(8)), a


def test_draws_are_in_range():
    for size in (1, 7, 1000, 10**6):
        idx = [draw_index(5, i, size) for i in range(512)]
        assert all(0 <= k < size for k in idx)
    assert set(draw_symmetry(5, i) for i in range(512)) == set(range(8))
