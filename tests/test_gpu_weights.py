"""GPU parity of a weight GENERATION (`Net::load`, network/mod.rs:16-35; reloaded before every move by
selfplay/src/main.rs:107): BatchNorm folding and the arrangement into the tensor core's shared-memory image happen
on the device (nn.cu `k_fold_weights`); the result must equal a plain f32 host restatement bit for bit, and a
generation swapped in between two moves must not disturb anything that is already enqueued."""
import numpy as np
import pytest

from oracle import net_ref
from oracle import oracle as O
from takzero_b200 import capi, network

from helpers import folded_layer, games_to_states

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype", [network.DTYPE_F16, network.DTYPE_BF16])
def test_device_fold_equals_host_restatement(dtype):
    n, blocks = 6, 2
    ref = net_ref.Net(n, seed=21, blocks=blocks, randomize_bn=True)
    t = ref.tensors()
    m = capi.BatchedMCTS(n, 4, 8, arena_slots=4096)
    network.set_weights(m, t, dtype)
    got = network.weight_set(m)
    hdr = got[:24].view(np.uint32)
    assert hdr[0] == 0x53575A54 and list(hdr[1:4]) == [n, blocks, 1 if dtype == network.DTYPE_F16 else 0]
    assert hdr[4] == 1  # first generation
    off = 256
    names = [("core.input_conv2d", "core.batch_norm", 64)]
    for b in range(blocks):
        for j in range(2):
            names.append((f"core.res_block_{b}.{j}.conv2d", f"core.res_block_{b}.{j}.batch_norm", 256))
    names.append(("policy.conv2d", None, 256))
    for conv_name, bn_name, cin_pad in names:
        bn = None if bn_name is None else tuple(t[f"{bn_name}.{f}"] for f in ("weight", "bias", "running_mean", "running_var"))
        cb = t.get(f"{conv_name}.bias")
        bits, bias = folded_layer(t[f"{conv_name}.weight"], bn, cb, cin_pad, dtype == network.DTYPE_F16)
        size = bits.size * 2
        assert np.array_equal(got[off:off + size].view(np.uint16), bits), conv_name
        off += size
        assert np.array_equal(got[off:off + 1024].view(np.uint32), bias.view(np.uint32)), conv_name + " bias"
        off += 1024
    heads = got[off:off + (512 + 76) * 4].view(np.float32)
    assert np.array_equal(heads[:256], t["value.conv2d.weight"].reshape(-1))
    assert np.array_equal(heads[256:512], t["ube.conv2d.weight"].reshape(-1))
    assert heads[512] == t["value.conv2d.bias"][0] and heads[513] == t["ube.conv2d.bias"][0]
    assert np.array_equal(heads[514:514 + n * n], t["value.linear.weight"].reshape(-1))
    assert np.array_equal(heads[550:550 + n * n], t["ube.linear.weight"].reshape(-1))
    assert heads[586] == t["value.linear.bias"][0] and heads[587] == t["ube.linear.bias"][0]
    m.close()


def test_generation_swap_between_moves():
    """tz_broadcast_weights without a communicator is Net::load on one GPU.  Generations alternate between the two
    weight sets: a move searched with network A, a reload to B between moves, a move with B, a reload back to A --
    every move equals the same move on a handle that only ever had that network, although the reloads are enqueued
    while the previous search may still be running (no host synchronisation in between)."""
    n, hk, G = 4, 4, 64
    nets = [net_ref.Net(n, seed=s, blocks=2, randomize_bn=True) for s in (1, 2)]
    games = [O.new_opening(n, hk, i % 8, i // 8 % 2) for i in range(G)]
    states = games_to_states(games)
    gum = np.random.default_rng(3).gumbel(size=(4, G, 256)).astype(np.float32)

    def play(handle, move_index):
        mv = handle.gumbel_sequential_halving(None, 8, 48, gum[move_index])
        handle.step(mv)
        return mv, handle.root_stats().copy()

    m = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    m.set_positions(states)
    network.broadcast_weights(m, nets[0].tensors())
    m.set_agent(capi.AGENT_NETWORK)
    got = []
    for i in range(4):
        if i > 0:
            network.broadcast_weights(m, nets[i % 2].tensors())
        got.append(play(m, i))
    gen, ms = network.weight_generation(m)
    assert gen == 4 and 0.0 < ms < 1000.0
    assert m.status() == 0
    m.close()
    # reference run: a fresh handle per network change, same positions carried over through the replayed moves
    r = capi.BatchedMCTS(n, hk, G, arena_slots=1 << 14)
    r.set_positions(states)
    network.set_weights(r, nets[0].tensors())
    r.set_agent(capi.AGENT_NETWORK)
    for i in range(4):
        if i > 0:
            network.set_weights(r, nets[i % 2].tensors())
            r.sync()  # the reference run waits for every reload; the run above never does
        mv, stats = play(r, i)
        assert np.array_equal(mv, got[i][0]), f"move {i}"
        assert np.array_equal(stats, got[i][1]), f"move {i} roots"
    r.close()


def test_broadcast_needs_tensors_on_the_root_and_checks_the_architecture():
    m = capi.BatchedMCTS(4, 4, 4, arena_slots=4096)
    with pytest.raises(capi.TakzeroError, match="root"):
        network.broadcast_weights(m, None)
    t = net_ref.Net(4, seed=1, blocks=2).tensors()
    with pytest.raises(capi.TakzeroError, match="residual blocks"):
        network.broadcast_weights(m, t, res_blocks=3)
    network.broadcast_weights(m, t, res_blocks=2)
    assert network.weight_generation(m)[0] == 1
    assert network.allreduce_sum(m, [5, 7]) == [5, 7]  # one rank: the sum is the value
    m.close()
