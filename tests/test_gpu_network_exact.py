"""The fused network (conv_tcgen05.cuh `k_conv3x3_pair`: input encoder, tower, policy convolution with the legal-logit
gather, head features; encode.cuh `warp_heads`) against float64 references, layer by layer.

* An EXACT network: sparse +-1 integer convolutions, integer biases, BatchNorm that folds to a scale of exactly 1.0,
  head 1x1 weights integers, head linear weights integers times a power of two.  Every activation is an integer and
  every f32 sum stays below 2^24, so f32 accumulation is exact in any order and the device output of a layer is the
  16-bit rounding of the exact value.  The integer reference below must then be matched bit for bit: legal logits,
  which are f32 sums, exactly; value and variance within 2 ulp of float64 tanh / exp (CUDA's tanhf / expf are
  accurate to 2 ulp).  This checks placement and indexing: the gather (also the whole-warp gather of squares with
  more than eight moves), packed and dense rows, chunks, bias, residual and the heads.
* Realistic weights (He-scaled, random BatchNorm): every layer read back from the device and compared with a float64
  convolution of the device's own 16-bit inputs under a rounding-error bound; the only check of the fractional input
  planes and of realistic rounding."""
import functools

import numpy as np
import pytest
import torch

from oracle import net_ref
from oracle import oracle as O
from takzero_b200 import capi, network

from helpers import (FILTERS, assert_tree_equal, folded_layer, games_to_states, random_playout_states,
                     to_bf16_bits)

pytestmark = pytest.mark.gpu

HK = 4
DTYPES = [network.DTYPE_F16, network.DTYPE_BF16]
# positions where one square has more than eight moves (the whole warp gathers them); in the 6x6 one squares 0, 5 and
# 30 all have 124 moves and are rows of the same epilogue warp
HEAVY = {6: "1212121,x4,1212121/x6/x6/x6/x6/1212121,x4,1212121 1 30",
         5: "12121212,x3,12121/x5/x5/x5/x5 1 30",
         4: "1212121,x3/x4/x4/x4 1 20"}
U = 2.0 ** -24  # unit roundoff of f32


@pytest.fixture(autouse=True)
def _device_matching_math():
    O.lib().tk_set_exact_math(1)
    yield
    O.lib().tk_set_exact_math(0)


# ---------------------------------------------------------------- 16-bit helpers


def round16(x, f16):
    """float64 -> the nearest value of the network's 16-bit type (round to nearest even), as float64."""
    if f16:
        return np.asarray(x, np.float64).astype(np.float16).astype(np.float64)
    return bits16_to_f64(to_bf16_bits(np.asarray(x, np.float64)), False)


def bits16_to_f64(bits, f16):
    if f16:
        return bits.view(np.float16).astype(np.float64)
    return (bits.astype(np.uint32) << np.uint32(16)).view(np.float32).astype(np.float64)


def ulp16(x, f16):
    """Spacing of the 16-bit type at |x| (subnormal spacing at and below the smallest normal)."""
    man, emin = (10, -14) if f16 else (7, -126)
    e = np.floor(np.log2(np.maximum(np.abs(x), 2.0 ** emin)))
    return 2.0 ** (e - man)


def ulps32(got, want):
    """|got - want| in units of the f32 spacing at want."""
    return np.abs(got.astype(np.float64) - want) / np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)


def unfold(bits, cin_pad, f16):
    """Inverse of folded_layer's arrangement: the device's 16-bit weights as float64 [256][cin_pad][3][3]."""
    blk = bits16_to_f64(bits, f16).reshape(cin_pad // 64, 9, 2, 8, 128, 8).transpose(2, 4, 0, 3, 5, 1)
    w = np.empty((FILTERS, cin_pad, 9))
    w[:, :, [4, 0, 1, 2, 3, 5, 6, 7, 8]] = blk.reshape(FILTERS, cin_pad, 9)
    return w.reshape(FILTERS, cin_pad, 3, 3)


def conv_layers(t, blocks):
    """(conv name, BatchNorm name or None, padded input channels) of every convolution, in launch order."""
    out = [("core.input_conv2d", "core.batch_norm", 64)]
    for b in range(blocks):
        for j in range(2):
            out.append((f"core.res_block_{b}.{j}.conv2d", f"core.res_block_{b}.{j}.batch_norm", 256))
    return out + [("policy.conv2d", None, 256)]


def device_weights(t, blocks, f16):
    """Per convolution: the folded 16-bit weights as float64 [256][cin_pad][3][3] and the f32 biases."""
    out = []
    for conv, bn, cin_pad in conv_layers(t, blocks):
        bnp = None if bn is None else tuple(t[f"{bn}.{f}"] for f in ("weight", "bias", "running_mean", "running_var"))
        bits, bias = folded_layer(t[f"{conv}.weight"], bnp, t.get(f"{conv}.bias"), cin_pad, f16)
        out.append((unfold(bits, cin_pad, f16), bias.astype(np.float64)))
    return out


# ---------------------------------------------------------------- positions


def pool(n, count, seed):
    """The heavy position first, then `count` - 1 positions of seeded random playouts (at least 4 plies in)."""
    rng = np.random.default_rng(seed)
    out = [O.from_tps(n, HK, HEAVY[n])]
    while len(out) < count:
        ps = random_playout_states(n, HK, int(rng.integers(1 << 30)), keep_terminal=False)[4:]
        for i in rng.choice(len(ps), size=min(3, len(ps)), replace=False):
            out.append(ps[int(i)])
    return out[:count]


def batch_slots(count, pool_size):
    """Pool index of every slot of a batch: the heavy position in slots 0 and 1 (their heavy squares share epilogue
    warps) and in every 37th slot, the others cycle through the pool."""
    idx = 1 + np.arange(count) % (pool_size - 1)
    idx[:2] = 0
    idx[::37] = 0
    return idx


def planes(games):
    n = games[0].n
    return np.stack([O.game_repr(g).reshape(-1, n, n) for g in games]).astype(np.float64)


# ---------------------------------------------------------------- part 1: the exact network


def sparse_conv(x, rows, n):
    """Integer 3x3 convolution with a sparse +-1 kernel: rows = (ci, ky, kx, sign) [256, nnz] each.  int64, exact."""
    ci, ky, kx, sign = rows
    xp = np.pad(x, ((0, 0), (0, 0), (1, 1), (1, 1)))
    i = np.arange(n)
    out = np.zeros((x.shape[0], FILTERS, n, n), np.int64)
    for s in range(0, x.shape[0], 16):
        g = xp[s:s + 16][:, ci[..., None, None], ky[..., None, None] + i[:, None], kx[..., None, None] + i[None, :]]
        out[s:s + 16] = (g * sign[..., None, None]).sum(axis=2)
    return out


def sparse_abs_conv(x, rows, n):
    return sparse_conv(np.abs(x), (rows[0], rows[1], rows[2], np.abs(rows[3])), n)


def draw_rows(rng, cin_ok, nnz, neg=0.5):
    """nnz distinct (input channel, tap) per output channel among the channels cin_ok, sign -1 with probability neg."""
    pick = np.argsort(rng.random((FILTERS, len(cin_ok) * 9)), axis=1)[:, :nnz]
    sign = np.where(rng.random(pick.shape) < neg, -1, 1)
    return (np.asarray(cin_ok)[pick // 9], (pick % 9) // 3, pick % 3, sign)


def dense(rows, cin):
    w = np.zeros((FILTERS, cin, 3, 3), np.float32)
    co = np.repeat(np.arange(FILTERS)[:, None], rows[0].shape[1], axis=1)
    w[co, rows[0], rows[1], rows[2]] = rows[3]
    return w


def integer_channels(n):
    """Input planes that only ever hold integers: all but my / the opponent's stones in reserve over their initial
    count and the flat-count difference over N^2 (repr.rs:199-227)."""
    c = 4 * n + 12
    return [i for i in range(c) if i not in (4 * n + 6, 4 * n + 8, 4 * n + 11)]


def grow_layer(rng, x, residual, cin_ok, n, neg0):
    """Greedy layer with rejection: the fewest negative weights (not fewer than the layer before, neg0), the most
    non-zeros per output channel (at most 12) and the highest share of active outputs (per-channel integer biases at
    a quantile of the sample) for which the activations of the sample stay <= 512 and at least 30 % of them are
    non-zero.  Without negative weights the residual stream of a deep tower only grows."""
    for neg in [v for v in (0.5, 0.7, 0.9) if v >= neg0]:
        for nnz in range(12, 0, -1):
            for share in (0.65, 0.5, 0.42):
                rows = draw_rows(rng, cin_ok, nnz, neg)
                pre = sparse_conv(x, rows, n) + (0 if residual is None else residual)
                per_channel = np.sort(pre.transpose(1, 0, 2, 3).reshape(FILTERS, -1), axis=1)
                at = np.rint((1.0 - rng.uniform(0.32, share, FILTERS)) * (per_channel.shape[1] - 1)).astype(int)
                bias = -per_channel[np.arange(FILTERS), at] + rng.integers(-2, 3, FILTERS)
                bias[bias == 0] = -1
                out = np.maximum(pre + bias[None, :, None, None], 0)
                if out.max() <= 512 and (out > 0).mean() >= 0.3:
                    return rows, bias.astype(np.float64), neg
    raise AssertionError("no layer keeps the activations <= 512 with density >= 30 %")


def head_calibration(rng, feats, lo, hi, nn):
    """Integer 1x1 conv bias and linear weights k * 2^-s, linear bias, so that the pre-activation of the sample
    positions spans [lo, hi]: feats [positions, squares] are the 1x1 convolution's outputs."""
    b1 = -float(np.round(np.median(feats)))
    k = rng.choice([-3, -2, -1, 1, 2, 3], size=nn)
    for sq in range(0, nn, 2):  # neighbours never share a weight (a swapped square index must show)
        if sq + 1 < nn and k[sq] == k[sq + 1]:
            k[sq + 1] = -k[sq + 1]
    raw = (np.maximum(feats + b1, 0) * k).sum(axis=1)
    q_lo, q_hi = np.quantile(raw, [0.03, 0.97])
    s = int(np.floor(np.log2(max(q_hi - q_lo, 1.0) / (hi - lo))))
    lin_b = float(np.round((lo + hi) / 2 * 2.0 ** s - (q_lo + q_hi) / 2)) * 2.0 ** -s
    return b1, (k * 2.0 ** -s).astype(np.float32), lin_b, 2.0 ** -s


class ExactNet:
    """The exact network of one board size and depth, and its reference on a pool of positions."""

    def __init__(self, n, blocks, pool_size, seed):
        self.n, self.blocks, nn = n, blocks, n * n
        rng = np.random.default_rng(seed)
        self.games = pool(n, pool_size, seed)
        self.states = games_to_states(self.games)
        self.actions = [O.possible_moves(g) for g in self.games]
        self.planes = planes(self.games)
        cin = self.planes.shape[1]
        ints = integer_channels(n)
        assert np.array_equal(self.planes[:, ints], np.round(self.planes[:, ints])), "integer input planes"
        ref = net_ref.Net(n, seed=seed, blocks=blocks)
        t = ref.tensors()
        sample = np.rint(self.planes[:64]).astype(np.int64)
        sample[:, [c for c in range(cin) if c not in ints]] = 0
        self.rows, self.bias = [], []
        x, neg = None, 0.5
        for li, (conv, bn, _) in enumerate(conv_layers(t, blocks)[:-1]):
            residual = x if li > 0 and li % 2 == 0 else None
            inp = sample if li == 0 else (x if li % 2 == 1 else t_act)
            rows, bias, neg = grow_layer(rng, inp, residual, ints if li == 0 else range(FILTERS), n, neg)
            out = np.maximum(sparse_conv(inp, rows, n) + bias[None, :, None, None].astype(np.int64) +
                             (0 if residual is None else residual), 0)
            out = np.rint(round16(out, True)).astype(np.int64)
            if li % 2 == 1:
                t_act = out
            else:
                x = out
            self.rows.append(rows)
            self.bias.append(bias)
            t[f"{conv}.weight"] = dense(rows, FILTERS if li else cin)
            t[f"{bn}.weight"] = np.ones(FILTERS, np.float32)
            t[f"{bn}.bias"] = bias.astype(np.float32)
            t[f"{bn}.running_mean"] = np.zeros(FILTERS, np.float32)
            t[f"{bn}.running_var"] = np.full(FILTERS, np.float32(1.0) - np.float32(1e-5), np.float32)
        cout = t["policy.conv2d.weight"].shape[0]
        self.rows.append(draw_rows(rng, range(FILTERS), 64))  # many terms: logits spread over many integers
        self.bias.append(rng.integers(-8, 9, FILTERS).astype(np.float64))
        t["policy.conv2d.weight"] = dense(self.rows[-1], FILTERS)[:cout]
        t["policy.conv2d.bias"] = self.bias[-1][:cout].astype(np.float32)
        self.cout = cout
        # heads: 1x1 weights +-1 on 24 channels, then calibrate on the sample's last-layer outputs
        pre_last = self._tower(sample, True)[1]
        self.head_grid = {}
        for head, (lo, hi) in (("value", (-4.0, 4.0)), ("ube", (-30.0, 5.0))):
            w1 = np.zeros(FILTERS, np.float32)
            w1[rng.choice(FILTERS, 24, replace=False)] = rng.choice([-1, 1], 24)
            feats = np.einsum("c,bcyx->byx", w1.astype(np.int64), pre_last).reshape(len(sample), nn)
            b1, lin, lin_b, self.head_grid[head] = head_calibration(rng, feats, lo, hi, nn)
            t[f"{head}.conv2d.weight"] = w1.reshape(1, FILTERS, 1, 1)
            t[f"{head}.conv2d.bias"] = np.array([b1], np.float32)
            t[f"{head}.linear.weight"] = lin.reshape(1, nn)
            t[f"{head}.linear.bias"] = np.array([lin_b], np.float32)
        self.tensors = t
        self.simhash = ref.simhash_matrix.numpy()
        self.seen = np.arange(pool_size) % 2 == 1  # marked seen with update_counts: local uncertainty 0
        self._refs = {}

    def _tower(self, x, f16):
        """Integer tower on planes x (integers; the fractional planes are multiplied by zero weights): the 16-bit
        outputs of every layer and the unrounded last one."""
        layers = []
        x = np.maximum(sparse_conv(x, self.rows[0], self.n) + self.bias[0][None, :, None, None].astype(np.int64), 0)
        x = np.rint(round16(x, f16)).astype(np.int64)
        layers.append(x)
        pre = x
        for b in range(self.blocks):
            tt = np.maximum(sparse_conv(x, self.rows[1 + 2 * b], self.n) +
                            self.bias[1 + 2 * b][None, :, None, None].astype(np.int64), 0)
            tt = np.rint(round16(tt, f16)).astype(np.int64)
            pre = np.maximum(sparse_conv(tt, self.rows[2 + 2 * b], self.n) +
                             self.bias[2 + 2 * b][None, :, None, None].astype(np.int64) + x, 0)
            x = np.rint(round16(pre, f16)).astype(np.int64)
            layers += [tt, x]
        return layers, pre

    def reference(self, dtype):
        """Per pool position: legal logits (possible_moves order), value, variance if unseen / seen, value and UBE
        pre-activations.  Asserts the preconditions of exactness on the pool before any GPU work."""
        if dtype in self._refs:
            return self._refs[dtype]
        f16 = dtype == network.DTYPE_F16
        n, nn, t = self.n, self.n * self.n, self.tensors
        x0 = np.rint(self.planes).astype(np.int64)
        x0[:, [c for c in range(x0.shape[1]) if c not in integer_channels(n)]] = 0
        # the device's fold of these weights is the integers themselves (BatchNorm scale exactly 1.0)
        folded = device_weights(t, self.blocks, f16)
        for li, ((w, b), rows, bias) in enumerate(zip(folded, self.rows, self.bias)):
            outs = self.cout if li == len(folded) - 1 else FILTERS
            want_w, want_b = dense(rows, w.shape[1]), bias.copy()
            want_w[outs:], want_b[outs:] = 0, 0
            assert np.array_equal(w, want_w) and np.array_equal(b, want_b), f"layer {li}: folded weights"
            taps = np.abs(w).sum(axis=(0, 1)).reshape(-1)
            kblocks = np.abs(w).reshape(FILTERS, -1, 64, 9).sum(axis=(0, 2, 3))
            assert (taps > 0).all() and (kblocks > 0).all(), "every tap and every k-block has weights"
        layers, pre_last = self._tower(x0, f16)
        ins = [x0] + layers[:-1]
        for li, (inp, out) in enumerate(zip(ins, layers)):
            rows, bias = self.rows[li], self.bias[li]
            resid = np.abs(layers[li - 2]) if li >= 2 and li % 2 == 0 else 0
            s = sparse_abs_conv(inp, rows, n) + np.abs(bias)[None, :, None, None] + resid
            assert s.max() < 2 ** 24, f"layer {li}: f32 sums exact"
            assert out.max() < 65504, f"layer {li}: no fp16 overflow"
            assert (out > 0).mean() >= 0.25, f"layer {li}: density {(out > 0).mean():.3f}"
        x = layers[-1]
        s = sparse_abs_conv(x, self.rows[-1], n) + np.abs(self.bias[-1])[None, :, None, None]
        assert s.max() < 2 ** 24, "policy convolution: f32 sums exact"
        policy = (sparse_conv(x, self.rows[-1], n) + self.bias[-1][None, :, None, None].astype(np.int64))
        policy = policy[:, : self.cout].reshape(len(x), -1)
        logits = []
        for p, acts in enumerate(self.actions):
            lg = policy[p, [O.move_index(n, a) for a in acts]].astype(np.float64)
            assert len(np.unique(lg)) >= len(acts) / 2, f"position {p}: distinct logits"
            logits.append(lg.astype(np.float32))
        pre = {}
        for head in ("value", "ube"):
            w1 = t[f"{head}.conv2d.weight"].reshape(-1).astype(np.int64)
            feats = np.einsum("c,bcyx->byx", w1, pre_last).reshape(len(x), nn)
            assert np.einsum("c,bcyx->byx", np.abs(w1), pre_last).max() < 2 ** 24, f"{head}: 1x1 sums exact"
            h = np.maximum(feats + float(t[f"{head}.conv2d.bias"][0]), 0)
            lin = t[f"{head}.linear.weight"].reshape(-1).astype(np.float64)
            lin_b = float(t[f"{head}.linear.bias"][0])
            grid = self.head_grid[head]  # every linear weight and the bias are integer multiples of it
            assert np.array_equal(lin / grid, np.round(lin / grid)) and lin_b / grid == round(lin_b / grid)
            assert ((np.abs(h * lin).sum(axis=1) + abs(lin_b)) / grid).max() < 2 ** 24, f"{head}: linear sums exact"
            pre[head] = (h * lin).sum(axis=1) + lin_b
        value = np.tanh(pre["value"])
        var_seen = np.minimum(np.maximum(np.exp(pre["ube"]), 0.0), 4.0)
        self._refs[dtype] = (logits, value, var_seen, pre)
        return self._refs[dtype]

    def check_coverage(self, dtype):
        """The value pre-activation spans [-4, 4] and the UBE pre-activation of the seen positions [-30, 5]."""
        _, _, _, pre = self.reference(dtype)
        v, u = pre["value"], pre["ube"][self.seen]
        assert v.min() <= -3.0 and v.max() >= 3.0 and (np.abs(v) < 1.0).any(), (v.min(), v.max())
        assert u.min() <= -25.0 and u.max() >= np.log(4.0) + 0.5, (u.min(), u.max())
        assert ((u > -20.0) & (u < np.log(4.0) - 0.1)).sum() >= 4, "seen positions with variances below 4"


@functools.lru_cache(maxsize=None)
def exact_net(n, blocks):
    return ExactNet(n, blocks, pool_size=96 if blocks == 3 else 48, seed=1000 * n + blocks)


def new_handle(net, count, dtype, **mode):
    m = capi.BatchedMCTS(net.n, HK, count, arena_slots=4096)
    if mode:
        network.debug_network_mode(m, **mode)
    network.set_weights(m, net.tensors, dtype)
    network.set_simhash(m, net.simhash)
    network.update_counts(m, net.states[net.seen])
    return m


def check_exact(net, dtype, count, **mode):
    logits_ref, value_ref, var_seen_ref, _ = net.reference(dtype)
    net.check_coverage(dtype)
    slots = batch_slots(count, len(net.games))
    m = new_handle(net, count, dtype, **mode)
    idx = network.simhash_indices(m, net.states)
    seen = np.isin(idx, idx[net.seen])  # a hash collision marks an unseen position as well
    assert seen[net.seen].all()
    logits, values, variances = network.evaluate(m, net.states[slots], [net.actions[i] for i in slots])
    assert m.status() == 0
    m.close()
    for q, p in enumerate(slots):
        bad = np.flatnonzero(logits[q] != logits_ref[p])
        assert bad.size == 0, (f"slot {q} (pool {p}): {bad.size} of {len(logits[q])} logits differ, first at move "
                               f"{O.move_str(net.actions[p][bad[0]])}: {logits[q][bad[0]]} != {logits_ref[p][bad[0]]}")
    du = ulps32(values, value_ref[slots])
    assert du.max() <= 2, f"value: {du.max()} ulp at slot {int(du.argmax())}"
    var_ref = np.where(seen[slots], var_seen_ref[slots], 4.0)
    du = ulps32(variances, var_ref)
    assert du.max() <= 2, f"variance: {du.max()} ulp at slot {int(du.argmax())}"


# ---------------------------------------------------------------- part 2: end-to-end sweep

SWEEP = [(4, c, {}) for c in (1, 9, 1184, 1185)] + [(5, c, {}) for c in (1, 5, 6, 740, 741, 801)] + \
        [(6, c, {}) for c in (1, 3, 4, 444, 445, 1000)] + \
        [(n, c, mode) for n, c in ((4, 1185), (5, 801), (6, 1000))
         for mode in ({"chunk_min_tiles": 3}, {"per_layer_launches": True})]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n,count,mode", SWEEP, ids=[f"{n}x{n}-{c}-{'-'.join(m) or 'fused'}" for n, c, m in SWEEP])
def test_exact_network_bit_exact(n, count, mode, dtype):
    """3 blocks.  4x4: the local chain and its limit (1184 positions); 5x5 / 6x6: packed rows, then dense rows with
    positions straddling tiles; the largest count of every board also in many chunks and one launch per layer.  The
    heavy position sits in slots 0, 1 and every 37th; half of the pool is marked seen (local uncertainty 0)."""
    check_exact(exact_net(n, 3), dtype, count, **mode)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n,blocks,count", [(6, 16, 445), (5, 20, 741), (6, 16, 96), (5, 20, 96)])
def test_exact_network_full_depth(n, blocks, count, dtype):
    check_exact(exact_net(n, blocks), dtype, count)


# ---------------------------------------------------------------- part 4: the queue paths


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [5, 6])
def test_root_expansion_logits_of_the_search_queue(n, dtype):
    """The search's own queue (k_select fills it, moves already grouped by square, no permutation): after the root
    expansion every root child carries the reference logit of its move."""
    net = exact_net(n, 3)
    logits_ref = net.reference(dtype)[0]
    G = len(net.games)
    m = capi.BatchedMCTS(n, HK, G, arena_slots=1 << 16)
    network.set_weights(m, net.tensors, dtype)
    m.set_positions(net.states)
    m.set_agent(capi.AGENT_NETWORK)
    m.simulate()
    assert m.status() == 0
    tbl, stats = m.root_children(), m.root_stats()
    for g in range(G):
        k = int(stats["n_children"][g])
        assert k == len(net.actions[g])
        want = dict(zip(net.actions[g], logits_ref[g]))
        got = tbl["logit"][g, :k]
        assert np.array_equal(got, np.array([want[int(mv)] for mv in tbl["moves"][g, :k]], np.float32)), f"game {g}"
    m.close()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("warps", [1, 8])
@pytest.mark.parametrize("n", [5, 6])
def test_single_tree_with_the_device_network(n, warps, dtype):
    """tei's path: k_tree_forward -> the network on 128 leaves (packed local chain) -> k_tree_backward, against the
    oracle's sequential tree whose agent evaluates the same weights through tz_evaluate on a second handle."""
    net = exact_net(n, 3)
    env = O.from_tps(n, HK, HEAVY[n]) if n == 6 else O.new_opening(n, HK, 5, 0)
    m = capi.BatchedMCTS(n, HK, 1, tree_batch=128, arena_slots=1 << 20)
    m.debug_tree_warps(warps)
    network.set_weights(m, net.tensors, dtype)
    m.set_agent(capi.AGENT_NETWORK)
    m.set_positions(games_to_states([env]))
    ev = capi.BatchedMCTS(n, HK, 128, arena_slots=4096)
    network.set_weights(ev, net.tensors, dtype)

    def agent(envs, acts):
        return network.evaluate(ev, games_to_states(envs), acts)

    cb = O.py_agent(agent)
    tree = O.Tree()
    for it in range(10):
        m.tree_simulate_batch(0.0, 128)
        tree.simulate_batch(cb, env, 0.0, 128)
        assert_tree_equal(m, tree, f"batch {it}")
    assert m.status() == 0
    for h in (m, ev):
        h.close()


# ---------------------------------------------------------------- part 3: realistic weights, layer by layer


def he_net(n, seed):
    ref = net_ref.Net(n, seed=seed, blocks=net_ref.res_blocks_for(n), randomize_bn=True)
    g = torch.Generator().manual_seed(seed + 2)
    with torch.no_grad():
        for mod in ref.modules():
            if isinstance(mod, torch.nn.Conv2d) and mod.kernel_size == (3, 3):
                fan_in = mod.weight.shape[1] * 9
                mod.weight.copy_(torch.randn(mod.weight.shape, generator=g) * np.sqrt(2.0 / fan_in))
    return ref


def conv64(x, w, dev):
    """float64 3x3 convolution, zero padding: x [B][cin][N][N], w [256][cin][3][3]."""
    xt = torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    wt = torch.from_numpy(np.ascontiguousarray(w)).to(dev)
    return torch.nn.functional.conv2d(xt, wt, padding=1).cpu().numpy()


def to_nchw(a, n):
    return np.ascontiguousarray(a.transpose(0, 2, 1).reshape(a.shape[0], a.shape[2], n, n)).astype(np.float64)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [4, 5, 6])
def test_every_layer_against_float64(n, dtype):
    """Full depth, He-scaled convolutions, random BatchNorm, 96 positions with the heavy one.  Every layer is read
    back (debug_layer_limit) and compared with a float64 convolution of the device's own 16-bit inputs, the folded
    16-bit weights and f32 biases (layer 0: the 16-bit planes the encoder produced).  Per element

        |y - ref| <= ulp16(ref) / 2 + 2 K 2^-24 S,   K = 9 cin_pad + 2,  S = sum |w x| + |b| + |residual|

    (round to 16 bits after f32 sums of K terms).  The legal logits (f32, no 16-bit rounding) are compared with the
    same term without the half ulp.  Value / variance: the f64 heads on the f64 pre-rounding last layer; the f32
    error of that layer (E, the bound above without the half ulp) propagates through the 1x1 convolution (256
    terms) and the linear layer (N^2 terms) as |dfeat| <= sum |w| E + 2 * 258 * 2^-24 sum |w f|, |dpre| <= sum |l|
    |dfeat| + 2 (N^2 + 2) 2^-24 sum |l h|, so |dvalue| <= (1 - tanh^2) |dpre| + 2 ulp and |dvariance| <= variance
    (e^|dpre| - 1) + 2 ulp (every position is marked seen, so the variance is clamp(exp(ube), 0, 4)).  The fraction
    of 16-bit outputs that differ from round16(ref) at all stays below MISMATCH[dtype]: 1e-2 for fp16, 1e-3 for bf16;
    measured on a B200 (1000 W): fp16 3.7e-3 .. 4.1e-3, bf16 3.3e-4 .. 3.6e-4."""
    f16 = dtype == network.DTYPE_F16
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    ref = he_net(n, 50 + n)
    t = ref.tensors()
    blocks = ref.core.blocks
    count = 96
    games = pool(n, count, 60 + n)
    actions = [O.possible_moves(g) for g in games]
    states = games_to_states(games)
    m = capi.BatchedMCTS(n, HK, count, arena_slots=4096)
    network.set_weights(m, t, dtype)
    network.set_simhash(m, ref.simhash_matrix.numpy())
    network.update_counts(m, states)  # every position seen: variance = clamp(exp(ube), 0, 4)
    logits, values, variances = network.evaluate(m, states, actions)
    planes16 = to_nchw(network.debug_activations(m, 2, count), n)
    assert np.array_equal(planes16[:, : planes(games).shape[1]], round16(planes(games), f16)), "encoder planes"
    xs, ts = [], []
    for b in range(blocks):
        network.debug_layer_limit(m, 2 * b + 2)
        network.evaluate(m, states, actions)
        xs.append(to_nchw(network.debug_activations(m, 0, count), n))
        ts.append(to_nchw(network.debug_activations(m, 1, count), n))
    network.debug_layer_limit(m, 2 * blocks + 1)
    network.evaluate(m, states, actions)
    xs.append(to_nchw(network.debug_activations(m, 0, count), n))
    assert m.status() == 0
    m.close()

    W = device_weights(t, blocks, f16)
    mism, total, worst = 0, 0, 0.0

    def check(li, inp, out, resid):
        nonlocal mism, total, worst
        w, b = W[li]
        r = 0.0 if resid is None else resid
        want = conv64(inp, w, dev) + b[None, :, None, None] + r
        s = conv64(np.abs(inp), np.abs(w), dev) + np.abs(b)[None, :, None, None] + np.abs(r)
        err32 = 2 * (9 * w.shape[1] + 2) * U * s
        y = np.maximum(want, 0.0)
        bound = 0.5 * ulp16(y + err32, f16) + err32
        excess = np.abs(out - y) - bound
        assert excess.max() <= 0, f"layer {li}: |y - ref| exceeds the bound by {excess.max():.3g}"
        mism += int((out != round16(y, f16)).sum())
        total += out.size
        worst = max(worst, float(np.abs(out).max()))
        return want, err32

    check(0, planes16, xs[0], None)
    for b in range(blocks):
        check(1 + 2 * b, xs[b], ts[b], None)
        pre_last, err_last = check(2 + 2 * b, ts[b], xs[b + 1], xs[b])
    frac = mism / total
    print(f"{n}x{n} {'fp16' if f16 else 'bf16'}: {frac:.3e} of the 16-bit outputs differ from round16(ref), "
          f"largest |activation| {worst:.4g}")
    assert frac <= MISMATCH[dtype]
    # policy convolution and the gather: f32 logits, no 16-bit rounding
    w, b = W[-1]
    pol = conv64(xs[-1], w, dev) + b[None, :, None, None]
    pol_s = conv64(np.abs(xs[-1]), np.abs(w), dev) + np.abs(b)[None, :, None, None]
    err = 2 * (9 * 256 + 2) * U * pol_s
    cout = t["policy.conv2d.weight"].shape[0]
    pol, err = pol[:, :cout].reshape(count, -1), err[:, :cout].reshape(count, -1)
    for q in range(count):
        idx = [O.move_index(n, a) for a in actions[q]]
        assert (np.abs(logits[q] - pol[q, idx]) <= err[q, idx]).all(), f"position {q}: logits"
    # heads from the f64 pre-rounding last layer
    f = np.maximum(pre_last, 0.0)
    nn = n * n
    pre = {}
    for head in ("value", "ube"):
        w1 = t[f"{head}.conv2d.weight"].reshape(-1).astype(np.float64)
        feat = np.einsum("c,bcyx->byx", w1, f).reshape(count, nn)
        dfeat = (np.einsum("c,bcyx->byx", np.abs(w1), err_last) +
                 2 * 258 * U * np.einsum("c,bcyx->byx", np.abs(w1), f)).reshape(count, nn)
        h = np.maximum(feat + float(t[f"{head}.conv2d.bias"][0]), 0.0)
        lin = t[f"{head}.linear.weight"].reshape(-1).astype(np.float64)
        p = (h * lin).sum(axis=1) + float(t[f"{head}.linear.bias"][0])
        dp = (np.abs(lin) * dfeat).sum(axis=1) + 2 * (nn + 2) * U * (np.abs(h * lin).sum(axis=1) + np.abs(p))
        pre[head] = (p, dp)
    p, dp = pre["value"]
    v = np.tanh(p)
    assert (np.abs(values - v) <= (1 - v * v) * dp + 2 * np.spacing(np.abs(v).astype(np.float32))).all(), "value"
    p, dp = pre["ube"]
    var = np.minimum(np.exp(p), 4.0)
    assert (np.abs(variances - var) <= var * np.expm1(dp) + 2 * np.spacing(var.astype(np.float32))).all(), "variance"


# Fraction of 16-bit layer outputs that differ from round16(float64 reference), about 2.5x the measured one.  Measured
# on an NVIDIA B200 (power limit 1000 W): fp16 3.7e-3 (4x4), 4.0e-3 (5x5), 4.1e-3 (6x6); bf16 3.3e-4, 3.6e-4, 3.5e-4.
# The largest |activation| of these towers was 1.1e4 (5x5), a factor 6 below fp16's largest finite value.
MISMATCH = {network.DTYPE_F16: 1e-2, network.DTYPE_BF16: 1e-3}
