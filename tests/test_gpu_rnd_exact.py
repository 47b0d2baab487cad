"""The RND local uncertainty of the 5x5 network (rnd.cu; net5.rs:120-146,193-211,271-277) against a float64 restatement,
on every path that uses it, and the input encoders on stacks taller than the encoding.

Raw space.  The device reports clamp((raw - min) / (max - min), 0, 1) * 4 combined as clamp(max(exp(ube), rnd), 0, 4).
With min = 0, max = M a little above the largest raw value and the UBE bias at -30 (exp(ube) < 1e-10), the variance is
4 raw / M up to one f32 rounding, so the device's raw value is variance * M / 4.

Error model (`rnd_reference`).  The six GEMMs run in TF32 tensor-op math: each operand carries a relative error of at
most u = 2^-10 (10 stored mantissa bits; truncation as well as rounding), products are accumulated in f32 in any order.
Per position, through the reference's own float64 activations, to first order:
  * an independent part: every product w x carries (d_w + d_x) with variance <= 2 u^2, the K-term f32 accumulation
    adds K (2^-24 sum |w x|)^2, the bias add (2^-24 v)^2; variances propagate through the later layers as
    var_out = var_in @ (W^2)^T on the units the ReLU passes; raw = sum d^2 with d = learning - target gets
    var(raw) = sum 4 d^2 (var_learning + var_target).  The bound takes SIGMAS = 6 standard deviations of it.
  * a common part: a rounding mode may shrink every product of one GEMM by the same relative amount (truncation does,
    by about 0.7 u), which no independence argument averages away.  Each GEMM gets |kappa| <= 2 u (and the input GEMM
    also the f32 error of the normalization x = p / sum p^2), and the bound adds sum |kappa| |d raw / d kappa|, the
    derivatives taken by forward-mode propagation.
  * the f32 finish (two bias adds, 512 squares, one division): 530 * 2^-24 raw.
The worst case sum |W| |x| is about sqrt(K) looser and would not tell a planted mistake from rounding.  An emulation of
TF32 truncation / rounding of these weight families on the CPU stays within 0.4 / 0.07 of this bound.

Measured on an NVIDIA B200 (power limit 1000 W), the largest |error| / bound (printed as "worst error / bound"):
position-dominant family 0.054 (3x3), 0.048 (4x4), 0.070 (5x5), 0.053 (6x6); default init 0.022, 0.026, 0.031, 0.025;
root expansion 0.062; tall stacks 0.054 .. 0.063.  Both network dtypes gave the same values."""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle import net_ref
from oracle import oracle as O
from takzero_b200 import capi, network, weights

from helpers import assert_roots_equal, games_to_states, oracle_children, random_playout_states, state_to_game, \
    states_equal

HK = {3: 0, 4: 4, 5: 4, 6: 4}
U_TF32 = 2.0 ** -10
U32 = 2.0 ** -24
SIGMAS = 6.0
NETS = ("rnd_learning", "rnd_target")
LAYERS = ("input_linear", "hidden_linear", "final_linear")
UBE_BIAS = -30.0
DTYPES = [network.DTYPE_F16, network.DTYPE_BF16]


@pytest.fixture(autouse=True)
def _device_matching_math():
    O.lib().tk_set_exact_math(1)
    yield
    O.lib().tk_set_exact_math(0)


# ---------------------------------------------------------------- reference


def rnd_reference(t, planes):
    """float64 `forward_rnd` (raw, before the normalization) of positions given as game_repr planes [P, C*N*N], and
    the error bound of the device's TF32 computation of it (module docstring).  Returns (raw [P], bound [P])."""
    p = np.asarray(planes, np.float64).reshape(len(planes), -1)
    x = p / (p * p).sum(axis=1, keepdims=True)
    eta = (p.shape[1] + 2) * U32
    out, var_out, tangents = {}, {}, {}
    for a in NETS:
        h, var = x, np.zeros_like(x)
        masks, ys = [], []
        for li, name in enumerate(LAYERS):
            W = t[f"{a}.{name}.weight"].astype(np.float64)
            b = t[f"{a}.{name}.bias"].astype(np.float64)
            W2 = W * W
            y = h @ W.T
            v = y + b
            var = (2 * U_TF32 ** 2 * ((h * h) @ W2.T) + var @ W2.T + W.shape[1] * (U32 * (np.abs(h) @ np.abs(W).T)) ** 2
                   + (U32 * v) ** 2)
            ys.append(y)
            if li < 2:
                masks.append(v > 0)
                h, var = np.where(masks[-1], v, 0.0), np.where(masks[-1], var, 0.0)
            else:
                out[a], var_out[a] = v, var
        for li in range(3):  # d outputs / d kappa of GEMM li: its product y, carried to the outputs
            tg = ys[li]
            for lj in range(li + 1, 3):
                tg = np.where(masks[lj - 1], tg, 0.0) @ t[f"{a}.{LAYERS[lj]}.weight"].astype(np.float64).T
            tangents[a, li] = tg
    d = out[NETS[0]] - out[NETS[1]]
    raw = (d * d).sum(axis=1)
    sigma = np.sqrt((4 * d * d * (var_out[NETS[0]] + var_out[NETS[1]])).sum(axis=1))
    common = np.zeros_like(raw)
    for (a, li), tg in tangents.items():
        common += (2 * U_TF32 + (eta if li == 0 else 0.0)) * np.abs(2 * (d * tg).sum(axis=1))
    return raw, SIGMAS * sigma + common + 530 * U32 * raw


def planes_of(games):
    return np.stack([O.game_repr(g) for g in games])


# ---------------------------------------------------------------- weights


def trunk_tensors(n, seed):
    """A small network of the board (1 residual block) with the RND pair in the reference's default nn.Linear init
    (family ii), the UBE bias at -30, min = 0, max = 1."""
    ref = net_ref.Net(n, seed=seed, blocks=1, rnd=True)
    t = ref.tensors()
    t["ube.linear.bias"] = np.array([UBE_BIAS], np.float32)
    return t


def position_dominant(t, seed):
    """Family (i): the input term dominates.  Learning: input weights N(0, 8^2) (with |x| ~ 0.1 .. 0.2 the input term
    has a standard deviation near 1, ten times the N(0, 0.1^2) biases), He-scaled N(0, 2/1024) hidden and final
    weights, hidden biases N(0, 0.1^2), final biases N(0, 3^2).  Target: the same with twice the gain in the first two
    layers, so the two networks are not exchangeable (a layer swapped between them changes raw).  Raw then varies
    widely between positions one move apart (the side to move swaps the plane groups)."""
    rng = np.random.default_rng(seed)
    t = dict(t)
    for a, gain in zip(NETS, (1.0, 2.0)):
        k = t[f"{a}.input_linear.weight"].shape[1]
        t[f"{a}.input_linear.weight"] = (rng.standard_normal((1024, k)) * 8.0 * gain).astype(np.float32)
        t[f"{a}.input_linear.bias"] = (rng.standard_normal(1024) * 0.1).astype(np.float32)
        t[f"{a}.hidden_linear.weight"] = (rng.standard_normal((1024, 1024)) * np.sqrt(2 / 1024) * gain).astype(np.float32)
        t[f"{a}.hidden_linear.bias"] = (rng.standard_normal(1024) * 0.1).astype(np.float32)
        t[f"{a}.final_linear.weight"] = (rng.standard_normal((512, 1024)) * np.sqrt(2 / 1024)).astype(np.float32)
        t[f"{a}.final_linear.bias"] = (rng.standard_normal(512) * 3.0).astype(np.float32)
    return t


FAMILIES = ("position-dominant", "default-init")


@functools.lru_cache(maxsize=None)
def family_tensors(n, family):
    t = trunk_tensors(n, 31 + n)
    return position_dominant(t, 70 + n) if family == FAMILIES[0] else t


def with_norm(t, lo, hi):
    t = dict(t)
    t["min"], t["max"] = np.array([lo], np.float32), np.array([hi], np.float32)
    return t


# ---------------------------------------------------------------- positions


def ply_pairs(n, count, seed):
    """`count` positions of seeded random playouts, in pairs one ply apart (positions 2i and 2i + 1), none finished."""
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < count:
        line = random_playout_states(n, HK[n], int(rng.integers(1 << 30)), keep_terminal=False)
        if len(line) >= 2:
            j = int(rng.integers(len(line) - 1))
            out += [line[j], line[j + 1]]
    return out[:count]


@functools.lru_cache(maxsize=None)
def pool(n, family, count):
    """Positions, their planes, float64 raw and bound, and M = max raw + bound, plus 5 %."""
    games = ply_pairs(n, count, 11 * n + count)
    pl = planes_of(games)
    raw, bound = rnd_reference(family_tensors(n, family), pl)
    return games, pl, raw, bound, float(np.float32(1.05 * (raw + bound).max()))


def device_raw(variance, M):
    return variance.astype(np.float64) * (M / 4.0)


def check_raw(got_var, raw, bound, M, what):
    """|device raw - float64 raw| <= bound (+ the f32 rounding of the normalization); returns the worst error / bound."""
    assert (got_var > 1e-6).all() and (got_var < 4.0).all(), f"{what}: variance outside (0, 4): RND does not decide"
    err = np.abs(device_raw(got_var, M) - raw)
    lim = bound + 4 * U32 * raw
    bad = np.flatnonzero(err > lim)
    assert bad.size == 0, (f"{what}: {bad.size} positions outside the bound, first slot {bad[0]}: raw {raw[bad[0]]:.6g} "
                           f"device {device_raw(got_var, M)[bad[0]]:.6g} bound {lim[bad[0]]:.3g}")
    return float((err / lim).max())


# ---------------------------------------------------------------- teeth (CPU)


@pytest.mark.parametrize("n", [5, 6])
def test_reference_bound_tells_planted_mistakes_from_rounding(n):
    """With the position-dominant family every planted mistake moves raw by at least 10x the bound on at least 80 % of
    the positions (zeroing the side-to-move plane: of the positions with black to move, where the plane is not
    already zero).  A device that made one of these mistakes cannot pass the sweep."""
    games, pl, raw, bound, _ = pool(n, FAMILIES[0], 200)
    t = family_tensors(n, FAMILIES[0])

    def moved(r2, on=slice(None)):
        share = float(np.mean((np.abs(r2 - raw) >= 10 * bound)[on]))
        return share

    mistakes = {}
    t2 = dict(t)
    t2["rnd_learning.final_linear.bias"] = np.zeros(512, np.float32)
    mistakes["drop a final bias"] = moved(rnd_reference(t2, pl)[0])
    mistakes["swap the rows of positions one ply apart"] = moved(raw.reshape(-1, 2)[:, ::-1].reshape(-1))
    p = pl.astype(np.float64)
    # x = p / sqrt(sum p^2) is what p * sqrt(sum p^2) gives under the reference's p / sum p^2
    mistakes["normalize by sqrt(sum p^2)"] = moved(rnd_reference(t, p * np.sqrt((p * p).sum(1, keepdims=True)))[0])
    cin = pl.shape[1] // (n * n)
    zeroed = pl.reshape(len(pl), cin, n * n).copy()
    zeroed[:, cin - 2] = 0.0
    black = np.array([g.to_move == 1 for g in games])
    assert 0.3 < black.mean() < 0.7
    mistakes["zero the side-to-move plane"] = moved(rnd_reference(t, zeroed.reshape(len(pl), -1))[0], black)
    t2 = dict(t)
    for f in ("weight", "bias"):
        t2[f"rnd_learning.hidden_linear.{f}"] = t[f"rnd_target.hidden_linear.{f}"]
        t2[f"rnd_target.hidden_linear.{f}"] = t[f"rnd_learning.hidden_linear.{f}"]
    mistakes["swap learning and target in the hidden layer"] = moved(rnd_reference(t2, pl)[0])
    print(f"{n}x{n}: bound / raw median {np.median(bound / raw):.3g}; share of positions moved by >= 10x the bound:",
          {k: round(v, 3) for k, v in mistakes.items()})
    for k, v in mistakes.items():
        assert v >= 0.8, f"{k}: only {v:.2f} of the positions move by 10x the bound"
    # raw really depends on the position: one ply changes it by far more than the bound
    assert np.median(np.abs(np.diff(raw.reshape(-1, 2), axis=1)).reshape(-1) / bound[::2]) > 20


def test_reference_matches_net_ref():
    """The float64 restatement computes what oracle/net_ref.py's f32 `normalized_rnd` computes (raw space)."""
    import torch

    n = 5
    ref = net_ref.Net(n, seed=3, blocks=1, rnd=True)
    games = ply_pairs(n, 40, 2)
    xs = torch.from_numpy(planes_of(games).reshape(len(games), ref.cin, n, n))
    with torch.no_grad():
        want = (ref.rnd_learning(xs) - ref.rnd_target(xs)).square().sum(dim=1).double().numpy()
    raw, bound = rnd_reference(ref.tensors(), planes_of(games))
    assert np.allclose(raw, want, rtol=1e-4, atol=0)
    assert (bound > 0).all() and (bound < 1e-2 * raw).all()


# ---------------------------------------------------------------- A: tz_evaluate sweep

SWEEP_COUNTS = {5: [1, 3, 4, 5, 31, 32, 33, 127, 128, 129, 1000], 3: [1, 33, 129], 4: [1, 33, 129], 6: [1, 33, 129]}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("n", [5, 3, 4, 6])
def test_rnd_sweep_against_float64(n, family, dtype):
    """Counts around the 4 warps of a CTA and the GEMM tiles; every slot holds its own position (shuffled per count),
    so a slot or row mix-up shows.  5x5 also evaluates count = Q on a handle whose Q (tree_batch) exceeds G."""
    counts = SWEEP_COUNTS[n]
    games, pl, raw, bound, M = pool(n, family, max(counts))
    t = with_norm(family_tensors(n, family), 0.0, M)
    states = games_to_states(games)
    actions = [O.possible_moves(g) for g in games]
    m = capi.BatchedMCTS(n, HK[n], max(counts), arena_slots=4096)
    network.set_weights(m, t, dtype)
    rng = np.random.default_rng(n)
    worst = 0.0
    for c in counts:
        idx = rng.permutation(len(games))[:c]
        _, _, var = network.evaluate(m, states[idx], [actions[i] for i in idx])
        worst = max(worst, check_raw(var, raw[idx], bound[idx], M, f"{n}x{n} {family} count {c}"))
    assert m.status() == 0
    m.close()
    if n == 5:
        q = capi.BatchedMCTS(n, HK[n], 8, tree_batch=300, arena_slots=4096)
        network.set_weights(q, t, dtype)
        idx = rng.permutation(len(games))[:300]
        _, _, var = network.evaluate(q, states[idx], [actions[i] for i in idx])
        worst = max(worst, check_raw(var, raw[idx], bound[idx], M, "count = Q > G"))
        assert q.status() == 0
        q.close()
    print(f"{n}x{n} {family} dtype {dtype}: worst error / bound {worst:.3f}, raw {raw.min():.4g} .. {raw.max():.4g}")


@pytest.mark.gpu
def test_rnd_clamp_edges_and_the_combine():
    """min / max inside the raw range: positions clearly below min give exactly 0 (exp(ube) underflows with the UBE
    bias at -200), clearly above max exactly 4.  Then the combine clamp(max(exp(ube), rnd), 0, 4) with exp(ube) of the
    device's own trunk (a second handle without RND, every position marked seen, reports clamp(exp(ube), 0, 4))."""
    n, family = 5, FAMILIES[0]
    games, pl, raw, bound, M = pool(n, family, 256)
    states, actions = games_to_states(games), [O.possible_moves(g) for g in games]
    lo, hi = (float(np.float32(q)) for q in np.quantile(raw, [0.3, 0.7]))
    t = with_norm(family_tensors(n, family), lo, hi)
    t["ube.linear.bias"] = np.array([-200.0], np.float32)
    m = capi.BatchedMCTS(n, HK[n], len(games), arena_slots=4096)
    network.set_weights(m, t)
    var = network.evaluate(m, states, actions)[2]
    below, above = raw + bound < lo, raw - bound > hi
    inside = ~below & ~above
    assert below.sum() >= 30 and above.sum() >= 30 and inside.sum() >= 30
    assert (var[below] == 0.0).all() and (var[above] == 4.0).all()
    want = (raw - lo) / (hi - lo) * 4.0
    assert (np.abs(var[inside] - want[inside]) <= (bound[inside] + 4 * U32 * raw[inside]) / (hi - lo) * 4.0 + 1e-6).all()
    # the combine: a UBE bias at log(median RND term) puts exp(ube) above the RND term on part of the positions; one of
    # 8 puts it above 4 everywhere (this trunk's UBE pre-activation without the bias stays within a few units of 0),
    # so the clamp at 4 decides
    t = with_norm(family_tensors(n, family), 0.0, M)
    trunk = {k: v for k, v in t.items() if not k.startswith("rnd_") and k not in ("min", "max")}
    rnd_var = 4.0 * raw / M
    for ube_bias, clamped in ((float(np.log(np.median(rnd_var))), False), (8.0, True)):
        t["ube.linear.bias"] = trunk["ube.linear.bias"] = np.array([ube_bias], np.float32)
        network.set_weights(m, t)
        var = network.evaluate(m, states, actions)[2]
        s = capi.BatchedMCTS(n, HK[n], len(games), arena_slots=4096)
        network.set_weights(s, trunk)
        network.set_simhash(s, np.zeros((s.input_channels * n * n, 32), np.float32))
        network.update_counts(s, states)
        ube_var = network.evaluate(s, states, actions)[2]  # clamp(exp(ube), 0, 4), the same trunk
        assert s.status() == 0
        s.close()
        slack = (bound + 4 * U32 * raw) / M * 4.0
        ube_wins, rnd_wins = ube_var > rnd_var + slack, ube_var < rnd_var - slack
        assert np.array_equal(var[ube_wins], ube_var[ube_wins])
        assert (np.abs(var[rnd_wins] - rnd_var[rnd_wins]) <= slack[rnd_wins] + 1e-7).all()
        if clamped:
            assert (ube_var == 4.0).all() and (var == 4.0).all(), "exp(ube) > 4: clamped to 4"
        else:
            assert ube_wins.sum() >= 10 and rnd_wins.sum() >= 10, (int(ube_wins.sum()), int(rnd_wins.sum()))
    assert m.status() == 0
    m.close()


# ---------------------------------------------------------------- B: search paths


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_root_expansion_std_dev_is_the_roots_own_rnd(dtype):
    """Batched simulate from fresh roots, 64 games, one already finished (it takes no queue slot, so the queue is one
    short of Q).  After the root's first visit every root child carries std_dev = sqrt(variance) of the root's own
    evaluation (kernels.cu expand_leaf_children: running std from 0 with one visit); each game's must be its own
    position's raw value within the bound."""
    n, family, G, finished_at = 5, FAMILIES[0], 64, 17
    games, pl, raw, bound, M = pool(n, family, 256)
    games, raw, bound = list(games[:G]), raw[:G].copy(), bound[:G].copy()
    done = random_playout_states(n, HK[n], 5)[-1]
    assert O.terminal(done) != O.T_NONE
    games[finished_at] = done
    m = capi.BatchedMCTS(n, HK[n], G, arena_slots=1 << 16)
    network.set_weights(m, with_norm(family_tensors(n, family), 0.0, M), dtype)
    m.set_agent(capi.AGENT_NETWORK)
    m.set_positions(games_to_states(games))
    m.simulate()
    assert m.status() == 0
    stats, tbl = m.root_stats(), m.root_children()
    live = np.arange(G) != finished_at
    std = stats["std_dev_bits"].view(np.float32)
    for g in np.flatnonzero(live):
        k = int(stats["n_children"][g])
        assert k > 0 and (tbl["std_dev"][g, :k].view(np.uint32) == stats["std_dev_bits"][g]).all(), f"game {g}"
    var = std[live].astype(np.float64) ** 2
    worst = check_raw(var.astype(np.float32), raw[live], bound[live] + 8 * U32 * raw[live], M, "root expansion")
    print(f"root expansion ({dtype}): worst error / bound {worst:.3f}")
    m.close()


# saturated mode: the learning network equals the target network except in the input columns of the pieces on these
# squares, so a position without a piece there has raw exactly 0 on every path (both networks do the same arithmetic
# on the same row), and one with such a piece a raw value far above the band.  With min / max a narrow band just above
# 0 the RND term is exactly 0 or 4 whatever the GEMMs' row count, which makes the search bit-exact comparable.
SAT_SQUARES = [6, 18]
SAT_LO, SAT_HI = 1.0, 1.001


@functools.lru_cache(maxsize=None)
def saturated_tensors():
    n = 5
    t = dict(family_tensors(n, FAMILIES[0]))
    cin, nn = 4 * n + 12, n * n
    for f in ("weight", "bias"):
        for name in LAYERS:
            t[f"rnd_learning.{name}.{f}"] = t[f"rnd_target.{name}.{f}"].copy()
    w = t["rnd_learning.input_linear.weight"].copy()
    rng = np.random.default_rng(9)
    for c in range(cin - 6):  # the piece planes: tops of both sides and the stack depths
        for sq in SAT_SQUARES:
            w[:, c * nn + sq] += (rng.standard_normal(1024) * 64.0).astype(np.float32)
    t["rnd_learning.input_linear.weight"] = w
    return with_norm(t, SAT_LO, SAT_HI)


def sat_columns():
    n, nn = 5, 25
    return np.array([c * nn + sq for c in range(4 * n + 12 - 6) for sq in SAT_SQUARES])


class SaturatedAgent:
    """The oracle side's agent: tz_evaluate of a second handle with the same weights.  Keeps every leaf's planes for
    the precondition check."""

    def __init__(self, dtype, capacity=128):
        self.ev = capi.BatchedMCTS(5, HK[5], capacity, arena_slots=4096)
        network.set_weights(self.ev, saturated_tensors(), dtype)
        self.planes = []
        self.cb = O.py_agent(self._evaluate)

    def _evaluate(self, envs, acts):
        self.planes += [O.game_repr(g) for g in envs]
        return network.evaluate(self.ev, games_to_states(envs), acts)

    def check(self, what):
        """Every leaf either has no piece on SAT_SQUARES (raw exactly 0) or lies above the band by more than the
        bound; both kinds occur.  Returns the leaf count."""
        pl = np.stack(self.planes)
        touched = (pl[:, sat_columns()] != 0).any(axis=1)
        raw, bound = rnd_reference(saturated_tensors(), pl[touched])
        assert (raw - bound > SAT_HI).all(), f"{what}: precondition: a leaf's raw lies within the bound of the band"
        assert 0.1 < touched.mean() < 0.9, f"{what}: {touched.mean():.2f} of the leaves have RND 4"
        assert self.ev.status() == 0
        print(f"{what}: {len(pl)} leaves, {int(touched.sum())} with RND 4, smallest margin "
              f"{float(((raw - bound) / SAT_HI).min()):.3g} x max")
        self.ev.close()
        return len(pl)


def sat_openings(count, seed):
    out = []
    for i in range(count):
        line = random_playout_states(5, HK[5], 1000 * seed + i, max_plies=6, keep_terminal=False)
        out.append(line[min(len(line) - 1, 2 + i % 4)])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_saturated_gumbel_search_equals_the_oracle(dtype):
    """Batched Gumbel sequential halving (k = 8, budget 48, 16 games, beta = 0.25) on the device network against the
    oracle's BatchedMCTS whose agent evaluates through tz_evaluate: every root and child bit for bit."""
    G = 16
    games = sat_openings(G, 1)
    agent = SaturatedAgent(dtype)
    m = capi.BatchedMCTS(5, HK[5], G, arena_slots=1 << 16)
    network.set_weights(m, saturated_tensors(), dtype)
    m.set_agent(capi.AGENT_NETWORK)
    m.set_positions(games_to_states(games))
    ob = O.Batched(games)
    rng = np.random.default_rng(3)
    betas = np.full(G, 0.25, np.float32)
    for move in range(2):
        gumbel = rng.gumbel(size=(G, m.move_stride)).astype(np.float32)
        got = m.gumbel_sequential_halving(betas, 8, 48, gumbel)
        want = ob.gumbel_sequential_halving(agent.cb, betas, 8, 48, gumbel)
        assert list(got) == want, f"move {move}: selected moves"
        assert_roots_equal(m, ob, f"move {move}")
        m.step(got)
        ob.step(want)
    assert m.status() == 0
    m.close()
    agent.check(f"Gumbel search ({dtype})")


@pytest.mark.gpu
@pytest.mark.parametrize("warps", [1, 8])
def test_saturated_single_tree_equals_the_oracle(warps):
    """tei's configuration: one game, tree_batch 128, 10 batches at beta = 0.25.  The first batch queues one leaf,
    so all but one queue slot are unwritten there; the RND pass must leave them alone.  The root has no piece on
    SAT_SQUARES: a piece there would give every leaf of the one tree RND 4."""
    env = next(g for g in sat_openings(12, 7) if not (planes_of([g])[0][sat_columns()] != 0).any())
    agent = SaturatedAgent(network.DTYPE_F16)
    m = capi.BatchedMCTS(5, HK[5], 1, tree_batch=128, arena_slots=1 << 20)
    m.debug_tree_warps(warps)
    network.set_weights(m, saturated_tensors(), network.DTYPE_F16)
    m.set_agent(capi.AGENT_NETWORK)
    m.set_positions(games_to_states([env]))
    tree = O.Tree()
    for it in range(10):
        m.tree_simulate_batch(0.25, 128)
        tree.simulate_batch(agent.cb, env, 0.25, 128)
        assert_game_equal(m, 0, tree.node, f"batch {it}")
    assert m.status() == 0
    m.close()
    agent.check(f"single tree ({warps} warps)")


@pytest.mark.gpu
def test_saturated_many_trees_equal_oracle_trees():
    """tz_trees_simulate_batch on 7 trees (16 leaves each, one network batch) against one oracle tree per game."""
    trees, batch = 7, 16
    envs = sat_openings(trees, 13)
    agent = SaturatedAgent(network.DTYPE_F16)
    m = capi.BatchedMCTS(5, HK[5], trees, tree_batch=trees * batch, arena_slots=1 << 18)
    network.set_weights(m, saturated_tensors(), network.DTYPE_F16)
    m.set_agent(capi.AGENT_NETWORK)
    m.set_positions(games_to_states(envs))
    oracle_trees = [O.Tree() for _ in range(trees)]
    for it in range(8):
        m.trees_simulate_batch(0.25, batch)
        for env, tree in zip(envs, oracle_trees):
            tree.simulate_batch(agent.cb, env, 0.25, batch)
        for g, tree in enumerate(oracle_trees):
            assert_game_equal(m, g, tree.node, f"batch {it} tree {g}")
    assert m.status() == 0
    m.close()
    agent.check("many trees")


def assert_game_equal(m, g, node, what):
    st, tbl = m.root_stats()[g], m.root_children()
    assert st["n_children"] == node.n_children and st["visit_count"] == node.visit_count, what
    assert (st["eval_tag"], st["eval_bits"]) == (node.evaluation.tag, node.evaluation.u.ply), what
    assert st["std_dev_bits"] == np.float32(node.std_dev).view(np.uint32), f"{what}: root std"
    oc, k = oracle_children(node), node.n_children
    for key in ("moves", "visits", "eval_tag", "eval_bits"):
        assert np.array_equal(tbl[key][g, :k], oc[key]), f"{what}: {key}"
    for key in ("logit", "prob", "std_dev"):
        assert np.array_equal(tbl[key][g, :k].view(np.uint32), oc[key].view(np.uint32)), f"{what}: {key}"


# ---------------------------------------------------------------- C: weight lifecycle


@pytest.mark.gpu
def test_rnd_weight_lifecycle(tmp_path):
    """load_model from a .ot; set_weights with a second RND model; a model without RND (4.0 everywhere); a model
    without min / max (defaults 0 and 1)."""
    n, count = 5, 64
    games, pl, raw, bound, M = pool(n, FAMILIES[0], 256)
    games, raw, bound = games[:count], raw[:count], bound[:count]
    states, actions = games_to_states(games), [O.possible_moves(g) for g in games]
    a = with_norm(family_tensors(n, FAMILIES[0]), 0.0, M)
    m = capi.BatchedMCTS(n, HK[n], count, arena_slots=4096)
    network.set_weights(m, a)
    var_a = network.evaluate(m, states, actions)[2]
    check_raw(var_a, raw, bound, M, "model A")
    weights.save_ot(str(tmp_path / "model_latest.ot"), a)
    f = capi.BatchedMCTS(n, HK[n], count, arena_slots=4096)
    network.load_model(f, str(tmp_path / "model_latest.ot"), allow_missing_set=True)
    assert np.array_equal(network.evaluate(f, states, actions)[2], var_a), "load_model"
    f.close()
    b = dict(family_tensors(n, FAMILIES[1]))
    raw_b, bound_b = rnd_reference(b, planes_of(games))
    mb = float(1.05 * (raw_b + bound_b).max())
    network.set_weights(m, with_norm(b, 0.0, mb))
    check_raw(network.evaluate(m, states, actions)[2], raw_b, bound_b, mb, "model B after A")
    network.set_weights(m, {k: v for k, v in a.items() if not k.startswith("rnd_")})
    assert (network.evaluate(m, states, actions)[2] == 4.0).all(), "a model without RND"
    assert raw_b.max() + bound_b.max() < 1.0
    network.set_weights(m, {k: v for k, v in b.items() if k not in ("min", "max")})
    check_raw(network.evaluate(m, states, actions)[2], raw_b, bound_b, 1.0, "default min 0, max 1")
    assert m.status() == 0
    m.close()


@pytest.mark.gpu
def test_broadcast_weights_without_a_communicator_equals_set_weights():
    """tz_broadcast_weights on a handle without a communicator is set_weights: the same outputs bit for bit, also
    after an earlier model with another estimator (set_weights A, then broadcast B gives B's), and a model without RND
    switches it off."""
    n, count = 5, 64
    games, pl, raw, bound, M = pool(n, FAMILIES[0], 256)
    states, actions = games_to_states(games[:count]), [O.possible_moves(g) for g in games[:count]]
    a = with_norm(family_tensors(n, FAMILIES[0]), 0.0, M)
    b = with_norm(position_dominant(trunk_tensors(n, 77), 78), 0.0, M)
    ref = capi.BatchedMCTS(n, HK[n], count, arena_slots=4096)
    out = {}
    for name, t in (("A", a), ("B", b)):
        network.set_weights(ref, t)
        out[name] = network.evaluate(ref, states, actions)
    assert not np.array_equal(out["A"][2], out["B"][2])
    m = capi.BatchedMCTS(n, HK[n], count, arena_slots=4096)
    network.broadcast_weights(m, a)
    for i in range(3):
        assert all(np.array_equal(x, y) for x, y in zip(network.evaluate(m, states, actions)[i], out["A"][i]))
    network.set_weights(m, a)
    network.broadcast_weights(m, b)
    got = network.evaluate(m, states, actions)
    assert np.array_equal(got[1], out["B"][1]), "value"
    assert np.array_equal(got[2], out["B"][2]), "variance: set_weights A, broadcast B must give B's estimator"
    network.broadcast_weights(m, {k: v for k, v in b.items() if not k.startswith("rnd_")})
    assert (network.evaluate(m, states, actions)[2] == 4.0).all(), "broadcast of a model without RND"
    assert m.status() == 0
    for h in (m, ref):
        h.close()


# ---------------------------------------------------------------- D: tall stacks

STONES = {3: 10, 4: 15, 5: 21, 6: 30}
CAPS = {3: 0, 4: 0, 5: 1, 6: 1}


def tall_stack_positions(n, seed):
    """One tall stack per position: heights 2N, 2N+1, 2N+2, 2N+3 and the largest the piece total allows (every stone
    of both sides, and a cap on top where the board has caps).  For each height, four colour patterns that agree
    everywhere except at depths 2N and 2N+1 below the top (the last encoded depth and the first one left out), flat,
    wall and cap tops, both sides to move, and 0 to 3 other pieces elsewhere.  Reserves are what the pieces on the
    board leave, so every position is one first_invalid_state accepts."""
    rng = np.random.default_rng(seed)
    S, Cp, nn = STONES[n], CAPS[n], n * n
    out = []
    for height in (2 * n, 2 * n + 1, 2 * n + 2, 2 * n + 3, 2 * S + Cp):
        for top in (0, 1, 2):
            if top == 2 and Cp == 0:
                continue
            if height == 2 * S + Cp and top != (2 if Cp else 0):
                continue
            for to_move in (0, 1):
                base = rng.integers(0, 2, height).astype(np.uint64)
                for flip in range(4):
                    colours = base.copy()
                    for bit, depth in ((1, 2 * n), (2, 2 * n + 1)):
                        if flip & bit and depth < height:
                            colours[height - 1 - depth] ^= np.uint64(1)
                    # keep each side within its stones (+ its cap on top)
                    top_colour = int(colours[-1])
                    owned = [int((colours == c).sum()) for c in (0, 1)]
                    limit = [S + (1 if top == 2 and c == top_colour else 0) for c in (0, 1)]
                    for c in (0, 1):
                        while owned[c] > limit[c]:
                            i = int(np.flatnonzero(colours[:-1] == c)[0])
                            colours[i] = np.uint64(1 - c)
                            owned = [int((colours == cc).sum()) for cc in (0, 1)]
                    if owned[0] > limit[0] or owned[1] > limit[1]:
                        continue
                    s = np.zeros((), capi.STATE_DTYPE)
                    sq = int(rng.integers(nn))
                    s["height"][sq] = height
                    s["stack"][sq] = int(sum(int(c) << i for i, c in enumerate(colours)))
                    s["top"][sq] = top
                    used = [owned[c] - (1 if top == 2 and c == top_colour else 0) for c in (0, 1)]
                    caps_used = [1 if top == 2 and c == top_colour else 0 for c in (0, 1)]
                    for other in rng.permutation(nn)[: int(rng.integers(4))]:
                        c = int(rng.integers(2))
                        if other == sq or used[c] >= S:
                            continue
                        s["height"][other], s["stack"][other], s["top"][other] = 1, c, 0
                        used[c] += 1
                    s["stones"] = [S - used[0], S - used[1]]
                    s["caps"] = [Cp - caps_used[0], Cp - caps_used[1]]
                    s["to_move"] = to_move
                    s["ply"] = int(s["height"].sum()) + 2
                    out.append(s.copy())
    states = np.array(out, dtype=capi.STATE_DTYPE)
    return states, [state_to_game(st, n, HK[n]) for st in states]


def tall_sets(n):
    states, games = tall_stack_positions(n, 400 + n)
    h = states["height"].max(axis=1)
    assert {2 * n, 2 * n + 1, 2 * n + 2, 2 * n + 3, 2 * STONES[n] + CAPS[n]} <= set(h.tolist())
    return states, games


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 4, 5, 6])
def test_tall_stacks_through_every_encoder_and_the_rules(n):
    """Against the oracle: tz_encode_planes bit for bit; the first convolution's input (debug_activations) as game_repr
    rounded to 16 bits, both dtypes; LCG-hash indices bit for bit; SimHash bits (which may differ only where the dot is
    within f32 rounding of 0); RND raw values within the bound; legal-move lists and order, terminal code, result and
    every legal move applied."""
    import torch

    states, games = tall_sets(n)
    count = len(games)
    cin = 4 * n + 12
    want = planes_of(games)
    m = capi.BatchedMCTS(n, HK[n], count, arena_slots=4096)
    got = network.encode_planes(m, states)
    assert np.array_equal(got.reshape(count, -1).view(np.uint32), want.view(np.uint32)), "tz_encode_planes"
    t = family_tensors(n, FAMILIES[0])
    raw, bound = rnd_reference(t, want)
    M = float(1.05 * (raw + bound).max())
    actions = [O.possible_moves(g) for g in games]
    worst = 0.0
    for dtype in DTYPES:
        network.set_weights(m, with_norm(t, 0.0, M), dtype)
        for lo in range(0, count, 96):  # the first convolution's read-back holds one chunk
            sl = slice(lo, min(lo + 96, count))
            k = sl.stop - sl.start
            _, _, var = network.evaluate(m, states[sl], actions[sl])
            worst = max(worst, check_raw(var, raw[sl], bound[sl], M, f"{n}x{n} tall stacks RND"))
            planes16 = network.debug_activations(m, 2, k)
            w = want[sl].reshape(k, cin, n * n).transpose(0, 2, 1)
            if dtype == network.DTYPE_F16:
                w16 = w.astype(np.float16).astype(np.float32)
            else:
                w16 = torch.from_numpy(np.ascontiguousarray(w)).to(torch.bfloat16).to(torch.float32).numpy()
            assert np.array_equal(planes16[:, :, :cin].view(np.uint32), w16.view(np.uint32)), "first convolution input"
            assert (planes16[:, :, cin:] == 0).all()
    ref = net_ref.Net(n, seed=4, blocks=1)
    xs = torch.from_numpy(want.reshape(count, cin, n, n))
    init = torch.empty(cin, n, n).uniform_(-100.0, 100.0, generator=torch.Generator().manual_seed(5))
    network.set_lcghash(m, init.numpy())
    assert np.array_equal(network.lcghash_indices(m, states), net_ref.Net.lcghash_indices(xs, init)), "LCG hash"
    matrix = ref.simhash_matrix.numpy()
    network.set_simhash(m, matrix)
    got_idx = network.simhash_indices(m, states)
    x = want.reshape(count, cin, n * n).astype(np.float64).copy()
    x[:, cin - 2] = 0.0
    x = x.reshape(count, -1)
    dots = x @ matrix.astype(np.float64)
    slack = 2 * x.shape[1] * U32 * (np.abs(x) @ np.abs(matrix.astype(np.float64)))
    want_bits = (dots >= 0)
    got_bits = ((got_idx[:, None] >> np.arange(32, dtype=np.uint32)) & 1).astype(bool)
    differ = got_bits != want_bits
    assert (np.abs(dots[differ]) <= slack[differ]).all(), "SimHash bits differ away from a zero dot"
    assert m.status() == 0
    m.close()
    # the rules
    h = capi.BatchedMCTS(n, HK[n], 4, arena_slots=4096)
    moves, counts = h.legal_moves(states)
    terms, results = h.result(states), h.game_result(states)
    chosen, src, expect = [], [], []
    for i, g in enumerate(games):
        tps = O.to_tps(g)
        assert terms[i] == O.terminal(g), f"terminal at {tps}"
        assert results[i] == O.lib().tk_game_result5(C.byref(g)), f"result at {tps}"
        legal = O.possible_moves(g)
        assert list(moves[i, :counts[i]]) == legal, f"legal moves at {tps}"
        for mv in legal:
            g2 = g.copy()
            O.play(g2, mv)
            chosen.append(mv)
            src.append(i)
            expect.append(g2)
    after, ok = h.apply(states[src], np.array(chosen, np.uint16))
    assert ok.all()
    want_after = games_to_states(expect)
    for j in range(len(chosen)):
        assert states_equal(after[j], want_after[j]), f"apply {O.move_str(chosen[j])} at {O.to_tps(games[src[j]])}"
    assert h.status() == 0
    h.close()
    print(f"{n}x{n}: {count} tall-stack positions, {len(chosen)} moves applied, {int((terms != 0).sum())} finished; "
          f"RND worst error / bound {worst:.3f}")
