"""GPU: training batches on the device (tz_target_buffer / tz_target_buffer_append / tz_training_batch).

Every example must equal what the Python restatement of the 8 symmetries (test_training_symmetry.py) and the oracle
make of the same target: planes = game_repr of the transformed position (and tz_encode_planes of it), policy / mask = a
scatter through move_index of the transformed moves.  The buffer fed by resident self-play must hold exactly the
targets tz_selfplay_read returns, without changing the search."""
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from takzero_b200 import build as tz_build
from takzero_b200 import capi, network
from test_training_symmetry import (REVERSIBLE_LIMIT, draw_index, draw_symmetry, output_channels, sym_move,
                                    sym_state)

pytestmark = pytest.mark.gpu

HK = 4
TARGET_KEYS = ("target_env", "target_value", "target_ube", "target_n", "target_offset", "policy_moves", "policy_probs")


def synthetic_targets(n, seed, count):
    """Targets of seeded playout positions (finished games included): random values and probabilities over the
    legal moves, in the layout tz_selfplay_read returns."""
    pp = O.playout_positions(n, HK, seed, 4, count, reversible_limit=REVERSIBLE_LIMIT)
    rng = np.random.default_rng(seed)
    counts = pp["n_moves"].astype(np.int32)
    offset = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.uint64)
    moves = np.concatenate([pp["moves"][i, :counts[i]] for i in range(count)]).astype(np.uint16)
    probs = np.concatenate([rng.dirichlet(np.ones(c)) if c else np.zeros(0) for c in counts]).astype(np.float32)
    return {"target_env": pp["states"].view(capi.STATE_DTYPE).reshape(count),
            "target_value": rng.uniform(-1, 1, count).astype(np.float32),
            "target_ube": rng.uniform(0, 4, count).astype(np.float32),
            "target_n": counts, "target_offset": offset, "policy_moves": moves, "policy_probs": probs}


def concat_targets(parts):
    out = {k: [] for k in TARGET_KEYS}
    base = 0
    for d in parts:
        for k in TARGET_KEYS:
            out[k].append(d[k] + np.uint64(base) if k == "target_offset" else d[k])
        base += len(d["policy_moves"])
    return {k: np.concatenate(v) if v else np.zeros(0) for k, v in out.items()}


def take(data, idx):
    """Targets idx of `data` as a new set in the same layout."""
    parts = []
    for i in idx:
        o, c = int(data["target_offset"][i]), int(data["target_n"][i])
        parts.append({"target_env": data["target_env"][i:i + 1], "target_value": data["target_value"][i:i + 1],
                      "target_ube": data["target_ube"][i:i + 1], "target_n": data["target_n"][i:i + 1],
                      "target_offset": np.zeros(1, np.uint64), "policy_moves": data["policy_moves"][o:o + c],
                      "policy_probs": data["policy_probs"][o:o + c]})
    return concat_targets(parts)


def expected_rows(n, data, i, t):
    """(policy, mask) rows [OC * N * N] of target i under symmetry t."""
    oc, nn = output_channels(n), n * n
    policy = np.zeros(oc * nn, np.float32)
    mask = np.zeros(oc * nn, np.uint8)
    o, c = int(data["target_offset"][i]), int(data["target_n"][i])
    for m, p in zip(data["policy_moves"][o:o + c], data["policy_probs"][o:o + c]):
        k = O.move_index(n, sym_move(t, n, int(m)))
        policy[k] = p
        mask[k] = 1
    return policy, mask


def batch_np(m, batch, seed=0, **kw):
    out = m.training_batch(batch, seed, **kw)
    return {k: v.cpu().numpy() for k, v in out.items()}


def check_batch(m, n, data, got, idx, sym):
    """The batch `got` against the restatement of targets idx under symmetries sym."""
    oc, nn = output_channels(n), n * n
    env = data["target_env"]
    states = np.stack([sym_state(int(t), n, env[i:i + 1].view(np.uint8)) for i, t in zip(idx, sym)])
    planes = got["planes"].reshape(len(idx), -1)
    want = network.encode_planes(m, states.view(capi.STATE_DTYPE).reshape(-1)).reshape(len(idx), -1)
    assert np.array_equal(planes.view(np.uint32), want.view(np.uint32)), "planes != tz_encode_planes"
    games = O.unpack_games(states, n, HK, REVERSIBLE_LIMIT)
    for b, (i, t) in enumerate(zip(idx, sym)):
        assert np.array_equal(planes[b].view(np.uint32), O.game_repr(games[b]).view(np.uint32)), (b, i, t)
        policy, mask = expected_rows(n, data, i, t)
        gp, gm = got["policy"][b].reshape(oc * nn), got["mask"][b].reshape(oc * nn)
        assert np.array_equal(gp.view(np.uint32), policy.view(np.uint32)), (b, i, t)
        assert np.array_equal(gm, mask), (b, i, t)
        o, c = int(data["target_offset"][i]), int(data["target_n"][i])
        assert int(gm.sum()) == c
        assert sorted(gp[gm == 1].tolist()) == sorted(data["policy_probs"][o:o + c].tolist())
        assert not gp[gm == 0].any()
    assert np.array_equal(got["value"].view(np.uint32), data["target_value"][idx].view(np.uint32))
    assert np.array_equal(got["ube"].view(np.uint32), data["target_ube"][idx].view(np.uint32))
    assert np.array_equal(got["index"], np.asarray(idx, np.int32))
    assert np.array_equal(got["symmetry"], np.asarray(sym, np.int32))


def ring(n, capacity, from_selfplay=False):
    m = capi.BatchedMCTS(n, HK, 4, arena_slots=4096)
    m.target_buffer(capacity, from_selfplay)
    return m


@pytest.mark.parametrize("n", [3, 4, 5, 6])
def test_explicit_examples_are_exact(n):
    data = synthetic_targets(n, 20 + n, 48)
    m = ring(n, 64)
    m.append_targets(data)
    assert m.target_buffer_info() == (48, 48)
    idx = np.repeat(np.arange(48), 8)
    sym = np.tile(np.arange(8), 48)
    got = batch_np(m, len(idx), indices=idx, symmetry=sym)
    check_batch(m, n, data, got, idx, sym)
    m.close()


@pytest.mark.parametrize("n", [4, 6])
def test_drawn_batches(n):
    data = synthetic_targets(n, 40 + n, 300)
    m = ring(n, 1000)
    m.append_targets(data)
    batch, seed = {4: 4096, 6: 2048}[n], 77  # one and two warps per example; the other tests use larger teams
    got = batch_np(m, batch, seed)
    assert got["index"].tolist() == [draw_index(seed, i, 300) for i in range(batch)]
    assert got["symmetry"].tolist() == [draw_symmetry(seed, i) for i in range(batch)]
    assert set(got["symmetry"].tolist()) == set(range(8))
    explicit = batch_np(m, batch, 5, indices=got["index"], symmetry=got["symmetry"])
    again = batch_np(m, batch, seed)
    for k in got:
        assert np.array_equal(explicit[k], got[k]), k
        assert np.array_equal(again[k], got[k]), k
    plain = batch_np(m, batch, seed, augment=False)
    assert np.array_equal(plain["index"], got["index"]) and not plain["symmetry"].any()
    check_batch(m, n, data, {k: v[:64] for k, v in got.items()}, got["index"][:64], got["symmetry"][:64])
    m.close()


def test_ring_wraps_and_rejects_bad_calls():
    import torch

    n = 4
    data = synthetic_targets(n, 3, 50)
    m = ring(n, 16)
    m.append_targets(take(data, range(10)))
    m.append_targets(take(data, range(10, 29)))  # 29 = capacity + 13: index 0 is the 14th target
    assert m.target_buffer_info() == (16, 29)
    got = batch_np(m, 16, indices=np.arange(16), symmetry=np.zeros(16))
    check_batch(m, n, take(data, range(13, 29)), got, np.arange(16), np.zeros(16, int))
    m.append_targets(take(data, range(29, 50)))  # more than the capacity in one call: the last 16 are kept
    assert m.target_buffer_info() == (16, 50)
    got = batch_np(m, 16, indices=np.arange(16), symmetry=np.zeros(16))
    check_batch(m, n, take(data, range(34, 50)), got, np.arange(16), np.zeros(16, int))
    before = batch_np(m, 16, indices=np.arange(16), symmetry=np.zeros(16))

    def rejected(fn, match):
        with pytest.raises(capi.TakzeroError, match=match):
            fn()
        assert m.target_buffer_info() == (16, 50)
        after = batch_np(m, 16, indices=np.arange(16), symmetry=np.zeros(16))
        for k in before:
            assert np.array_equal(after[k], before[k]), k

    bad = take(data, range(3))
    too_many = dict(bad, target_n=np.array([1, m.move_stride + 1, 1], np.int32))
    rejected(lambda: m.append_targets(too_many), "move_stride")
    outside = dict(bad, target_offset=np.array([0, 0, len(bad["policy_moves"]) - 1], np.uint64))
    rejected(lambda: m.append_targets(outside), "outside")
    for move in (0x0004 | (4 << 3), 3 << 6, (0x80 | 0x01) << 8, 0xF0 << 8):  # off board, piece 3, pattern bits
        wrong = dict(bad, policy_moves=bad["policy_moves"].copy())
        wrong["policy_moves"][-1] = move
        rejected(lambda: m.append_targets(wrong), "move_index")
    twice = dict(bad, policy_moves=bad["policy_moves"].copy())
    last = int(bad["target_offset"][-1])
    twice["policy_moves"][last + 1] = twice["policy_moves"][last]
    rejected(lambda: m.append_targets(twice), "twice")
    rejected(lambda: batch_np(m, 4, indices=[0, 1, 16, 2]), "size")
    rejected(lambda: batch_np(m, 2, symmetry=[0, 8]), "0..7")
    rejected(lambda: m.training_batch(0, 1), "batch")
    host = TrainingOutputsOnHost(m, 4)
    rejected(host.call, "device memory")
    if torch.cuda.device_count() > 1:
        other = {"value": torch.empty(4, dtype=torch.float32, device="cuda:1")}
        with pytest.raises(ValueError):
            m.training_batch(4, 1, out=other)
    # capacity 0 frees the buffer; a new buffer replaces the old one and starts empty
    m.target_buffer(0)
    with pytest.raises(capi.TakzeroError, match="no target buffer"):
        m.target_buffer_info()
    with pytest.raises(capi.TakzeroError, match="no target buffer"):
        m.append_targets(bad)
    m.target_buffer(8)
    assert m.target_buffer_info() == (0, 0)
    with pytest.raises(capi.TakzeroError, match="empty"):
        m.training_batch(1, 1)
    m.target_buffer(8)
    m.append_targets(bad)
    assert m.target_buffer_info() == (3, 3)
    m.close()


class TrainingOutputsOnHost:
    """tz_training_batch with a host pointer among the outputs."""

    def __init__(self, m, batch):
        self.m, self.batch = m, batch
        self.host = np.zeros(batch, np.float32)

    def call(self):
        import ctypes as C

        p = capi.TrainingBatchParams(self.batch, None, None, 1, 1, None, None, None,
                                     self.host.ctypes.data_as(C.c_void_p).value, None, None, None)
        capi._check(capi.lib().tz_training_batch(self.m.handle, C.byref(p)))


def _params(k, budget, seed, beta=0.0):
    steps = k.bit_length() - 1
    vis = float(budget // steps // k * ((1 << steps) - 1))
    return capi.SelfplayParams(k, budget, beta, 10, 32, 0.5, vis, 0.25, seed)


def _selfplay_handle(n, G, seed):
    m = capi.BatchedMCTS(n, HK, G, arena_slots=1 << 15)
    m.new_openings(seed=seed)
    return m


@pytest.mark.parametrize("case", ["plain", "exploration", "queue_full"])
def test_buffer_fed_by_selfplay_holds_the_read_targets(case):
    n, G, k, budget, moves, seed = 4, 32, 8, 48, 70, 3
    beta = 0.5 if case == "exploration" else 0.0
    out_bytes = 64 << 10 if case == "queue_full" else 0
    read_every = 12 if case == "queue_full" else 1
    fed, plain, unfed = (_selfplay_handle(n, G, seed) for _ in range(3))
    capacity = 100 if case == "queue_full" else 400
    fed.target_buffer(capacity, from_selfplay=True)
    unfed.target_buffer(capacity, from_selfplay=False)
    for m in (fed, plain, unfed):
        m.selfplay_record(True, output_bytes=out_bytes)
    sp = _params(k, budget, seed, beta)
    reads = []
    for step in range(moves):
        for m in (fed, plain, unfed):
            m.selfplay_move(sp)
        if (step + 1) % read_every == 0 or step == moves - 1:
            got = [m.selfplay_read() for m in (fed, plain, unfed)]
            for d in got[1:]:
                for key in TARGET_KEYS + ("replay_start", "replay_moves", "replay_game"):
                    assert d[key].tobytes() == got[0][key].tobytes(), key
            reads.append(got[0])
    for m in (plain, unfed):
        assert m.positions().tobytes() == fed.positions().tobytes()
        ch, ref = m.root_children(), fed.root_children()
        for key in ref:
            assert np.array_equal(ch[key], ref[key]), key
        c, r = m.counters(), fed.counters()
        assert (c.simulations, c.evaluations, c.known, c.expansions) == (r.simulations, r.evaluations, r.known,
                                                                           r.expansions)
        assert m.status() == fed.status()
    if case == "queue_full":
        assert fed.status() & capi.STATUS_TARGETS_FULL
    assert unfed.launch_count() == plain.launch_count()
    assert fed.launch_count() == plain.launch_count() + moves
    assert unfed.target_buffer_info() == (0, 0)
    data = concat_targets(reads)
    total = len(data["target_value"])
    assert total > capacity, "the ring wraps"
    size, appended = fed.target_buffer_info()
    assert (size, appended) == (capacity, total)
    idx = np.arange(size)
    got = batch_np(fed, size, indices=idx, symmetry=np.zeros(size))
    check_batch(fed, n, take(data, range(total - size, total)), got, idx, np.zeros(size, int))
    for m in (fed, plain, unfed):
        m.close()


DRIVER = r'''
#include <cuda_runtime.h>
#include <cstdio>
#include <fstream>
#include "takzero_b200.hpp"
using namespace takzero;
// argv: targets file, board size, half komi, output file.  Parses every line with Target::parse, appends them with
// BatchedMCTS::append_targets and writes the identity batch over every index: planes, policy, mask, value, ube.
int main(int argc, char** argv) {
    const int n = atoi(argv[2]), hk = atoi(argv[3]);
    std::ifstream in(argv[1]);
    std::vector<Target> targets;
    for (std::string line; std::getline(in, line);) {
        Target t;
        if (!Target::parse(line, n, &t)) return 3;
        targets.push_back(t);
    }
    BatchedMCTS m(n, hk, 1, 0, 0, 4096);
    m.target_buffer(targets.size());
    m.append_targets(targets);
    const int B = (int)targets.size(), nn = n * n, C = 2 * (2 * n + 5) + 2, OC = 3 + 4 * ((1 << n) - 2);
    std::vector<uint64_t> idx(B);
    std::vector<int> sym(B, 0);
    for (int i = 0; i < B; i++) idx[i] = i;
    const size_t sizes[5] = {(size_t)B * C * nn * 4, (size_t)B * OC * nn * 4, (size_t)B * OC * nn, (size_t)B * 4,
                             (size_t)B * 4};
    void* d[5];
    for (int i = 0; i < 5; i++) cudaMalloc(&d[i], sizes[i]);
    tz_training_batch_t p{};
    p.batch = B;
    p.indices = idx.data();
    p.symmetry = sym.data();
    p.planes = (float*)d[0];
    p.policy = (float*)d[1];
    p.mask = (uint8_t*)d[2];
    p.value = (float*)d[3];
    p.ube = (float*)d[4];
    m.training_batch(p);
    check(tz_sync(m.handle()));
    FILE* f = fopen(argv[4], "wb");
    for (int i = 0; i < 5; i++) {
        std::vector<char> h(sizes[i]);
        cudaMemcpy(h.data(), d[i], sizes[i], cudaMemcpyDeviceToHost);
        fwrite(h.data(), 1, sizes[i], f);
        cudaFree(d[i]);
    }
    fclose(f);
    printf("%d\n", B);
    return 0;
}
'''


def test_cpp_append_of_a_targets_file_equals_the_read_arrays(tmp_path):
    tz_build.build()
    libdir = os.path.dirname(capi.LIB_PATH)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src, exe = tmp_path / "driver.cpp", tmp_path / "driver"
    src.write_text(DRIVER)
    cuda = "/usr/local/cuda"
    subprocess.check_call(["g++", "-std=c++17", "-O1", str(src), "-o", str(exe), f"-I{root}/include",
                           f"-I{cuda}/include", f"-L{libdir}", "-ltakzero_b200", f"-L{cuda}/lib64", "-lcudart",
                           f"-Wl,-rpath,{libdir}", f"-Wl,-rpath,{cuda}/lib64"])
    n, G, k, budget, moves, seed = 4, 32, 8, 48, 50, 5
    run = tmp_path / "run"
    run.mkdir()
    flags = ["--board", str(n), "--half-komi", str(HK), "--games", str(G), "--sampled-actions", str(k), "--budget",
             str(budget), "--moves", str(moves), "--seed", str(seed), "--arena-slots", str(1 << 15), "--resident"]
    out = subprocess.run([os.path.join(libdir, "bin", "selfplay"), "--directory", str(run), *flags],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr
    out = subprocess.run([str(exe), str(run / "targets-selfplay.txt"), str(n), str(HK), str(tmp_path / "cpp.bin")],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    count = int(out.stdout.split()[0])
    # the same self-play through the Python binding, its read arrays appended as they are
    m = _selfplay_handle(n, G, seed)
    m.selfplay_record(True)
    sp = _params(k, budget, seed)
    reads = []
    for _ in range(moves):
        m.selfplay_move(sp)
        reads.append(m.selfplay_read())
    data = concat_targets(reads)
    assert len(data["target_value"]) == count > 0
    m.target_buffer(count)
    m.append_targets(data)
    got = batch_np(m, count, indices=np.arange(count), symmetry=np.zeros(count))
    want = b"".join(got[k].tobytes() for k in ("planes", "policy", "mask", "value", "ube"))
    assert (tmp_path / "cpp.bin").read_bytes() == want
    m.close()
