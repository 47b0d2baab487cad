"""GPU: the novelty set as part of a generation (tz_update_counts_buffer / tz_broadcast_novelty_set).

Marking a training batch on the device must set exactly the bits that tz_update_counts sets for the same targets,
transformed on the host with the restated symmetries of test_training_symmetry.py, and exactly for the (index,
symmetry) pairs tz_training_batch uses with the same params.  A set generation must be indistinguishable from
tz_set_simhash with the same image -- for the search, its targets and tz_evaluate -- whatever the image's source, and
it must take effect between the moves enqueued before and after it.  Two ranks (skipped on fewer than two GPUs) must
end with the root's set, and a rank with another hash must flag the mismatch and keep its set.  Every comparison is
bit for bit."""
import ctypes as C
import hashlib
import os
import socket

import numpy as np
import pytest
import torch

from takzero_b200 import capi, network, weights
from test_gpu_training_batch import HK, synthetic_targets
from test_training_symmetry import sym_state

pytestmark = pytest.mark.gpu

SET_BYTES = 1 << 29
EINVAL, ENOWEIGHTS = -1, -5  # TZ_EINVAL, TZ_ENOWEIGHTS
STATUS_WEIGHTS_MISMATCH = 512


def hash_inputs(n, kind, seed):
    """(SimHash matrix or LCG multipliers) for an n x n handle."""
    cin = 2 * (2 * n + 5) + 2
    rng = np.random.default_rng(seed)
    if kind == "simhash":
        return rng.standard_normal((cin * n * n, 32)).astype(np.float32)
    return rng.uniform(-100.0, 100.0, (cin, n, n)).astype(np.float32)


def set_hash(m, kind, w, bitset=None):
    (network.set_simhash if kind == "simhash" else network.set_lcghash)(m, w, bitset)


def hashed(n, kind, w, games=4, bitset=None, capacity=0):
    m = capi.BatchedMCTS(n, HK, games, arena_slots=4096)
    network.set_weights(m, weights.random_init(n, seed=3, blocks=1))
    set_hash(m, kind, w, bitset)
    if capacity:
        m.target_buffer(capacity)
    return m


def kept(data, appended, capacity):
    """Positions the ring keeps, oldest first (index 0 of tz_training_batch)."""
    first = max(0, appended - capacity)
    return data["target_env"][first:appended]


def host_marked(n, kind, w, env, idx, sym, bitset=None):
    """The image tz_update_counts gives for targets idx under symmetries sym."""
    states = np.stack([sym_state(int(t), n, env[int(i):int(i) + 1].view(np.uint8)) for i, t in zip(idx, sym)])
    b = hashed(n, kind, w, bitset=bitset)
    network.update_counts(b, states.view(capi.STATE_DTYPE).reshape(-1))
    image = network.read_novelty_set(b)
    b.close()
    return image


def mark_rc(m, batch, indices=None, symmetry=None, augment=0, seed=0):
    idx = None if indices is None else np.ascontiguousarray(indices, np.uint64)
    sym = None if symmetry is None else np.ascontiguousarray(symmetry, np.int32)
    p = capi.TrainingBatchParams(batch, capi._ptr(idx), capi._ptr(sym), augment, seed)
    return capi.lib().tz_update_counts_buffer(m.handle, C.byref(p))


@pytest.mark.parametrize("n,kind", [(6, "simhash"), (4, "lcghash")])
def test_marking_equals_the_host_path(n, kind):
    w = hash_inputs(n, kind, 11)
    data = synthetic_targets(n, 30 + n, 64)
    cap = 40  # 64 appended into 40 slots: the ring has wrapped
    env = kept(data, 64, cap)
    rng = np.random.default_rng(n)
    explicit = (80, dict(indices=rng.integers(0, cap, 80), symmetry=rng.integers(0, 8, 80)))
    for batch, kw in [explicit, (64, dict(augment=True)), (50, dict(augment=False))]:
        m = hashed(n, kind, w, capacity=cap)
        m.append_targets(data)
        seed = 7 + batch
        out = m.training_batch(batch, seed, **kw)
        idx, sym = out["index"].cpu().numpy(), out["symmetry"].cpu().numpy()
        if "indices" in kw:
            assert np.array_equal(idx, kw["indices"]) and np.array_equal(sym, kw["symmetry"])
        if kw.get("augment") is False:
            assert not sym.any()
        m.update_counts_buffer(batch, seed, **kw)
        got = network.read_novelty_set(m)
        want = host_marked(n, kind, w, env, idx, sym)
        assert np.array_equal(got, want), (n, kind, batch, kw.keys())
        assert np.unpackbits(got[got != 0]).sum() >= len(set(zip(idx.tolist(), sym.tolist()))) // 2
        # marking the same batch again changes nothing
        m.update_counts_buffer(batch, seed, **kw)
        assert np.array_equal(network.read_novelty_set(m), want)
        m.close()


def test_rejections_leave_the_set_unchanged():
    n, kind = 6, "simhash"
    w = hash_inputs(n, kind, 12)
    data = synthetic_targets(n, 41, 24)
    m = hashed(n, kind, w, capacity=32)
    m.append_targets(data)
    m.update_counts_buffer(16, 5)
    before = network.read_novelty_set(m)
    assert mark_rc(m, 4, indices=[0, 1, 24, 2]) == EINVAL
    assert mark_rc(m, 3, symmetry=[0, 8, 1]) == EINVAL
    assert mark_rc(m, 2, symmetry=[-1, 0]) == EINVAL
    assert mark_rc(m, 0) == EINVAL
    assert mark_rc(m, -3) == EINVAL
    m.sync()
    assert np.array_equal(network.read_novelty_set(m), before)
    m.close()
    # an empty buffer, no buffer, and no hash
    empty = hashed(n, kind, w, capacity=8)
    assert mark_rc(empty, 4, augment=1) == EINVAL
    assert not network.read_novelty_set(empty).any()
    empty.target_buffer(0)
    assert mark_rc(empty, 4, augment=1) == EINVAL
    empty.close()
    nohash = capi.BatchedMCTS(n, HK, 4, arena_slots=4096)
    network.set_weights(nohash, weights.random_init(n, seed=3, blocks=1))
    nohash.target_buffer(32)
    nohash.append_targets(data)
    assert mark_rc(nohash, 4, augment=1) == ENOWEIGHTS
    nohash.close()


# ---- set generations ---------------------------------------------------------------------------------------------

def selfplay_params(seed):
    k, budget = 8, 48
    vis = float(budget // 3 // k * 7)
    return capi.SelfplayParams(k, budget, 0.5, 10, 32, 0.5, vis, 0.25, seed)  # exploration half: variance matters


def search_handle(w, bitset=None):
    n, G = 6, 16
    m = capi.BatchedMCTS(n, HK, G, arena_slots=1 << 15)
    network.set_weights(m, weights.random_init(n, seed=8, blocks=2))
    m.set_agent(capi.AGENT_NETWORK)
    network.set_simhash(m, w, bitset)
    m.selfplay_record(True)
    m.new_openings(seed=4)
    return m


def run(m, moves, seed0):
    roots = []
    for i in range(moves):
        m.selfplay_move(selfplay_params(seed0 + i))
        roots.append(m.root_children())
    return roots


def same_run(a, b, roots_a, roots_b):
    for ra, rb in zip(roots_a, roots_b):
        for key in ra:
            assert np.array_equal(np.asarray(ra[key]), np.asarray(rb[key])), key
    da, db = a.selfplay_read(), b.selfplay_read()
    assert da["n_targets"] == db["n_targets"]
    for key in da:
        if isinstance(da[key], np.ndarray):
            assert np.array_equal(da[key].view(np.uint8), db[key].view(np.uint8)), key
    states = a.positions()
    actions = [[] for _ in states]
    assert np.array_equal(network.evaluate(a, states, actions)[2].view(np.uint32),
                          network.evaluate(b, states, actions)[2].view(np.uint32))
    assert np.array_equal(network.read_novelty_set(a), network.read_novelty_set(b))


def random_image(seed):
    return np.random.default_rng(seed).integers(0, 256, SET_BYTES, dtype=np.uint8)


@pytest.mark.parametrize("source", ["pinned", "pageable", "null_after_marks"])
def test_set_generation_equals_set_simhash(source):
    n, kind = 6, "simhash"
    w = hash_inputs(n, kind, 21)
    image = random_image(5)
    if source == "null_after_marks":
        # the root's own set after device marks: the reference applies the same marks on the host
        data = synthetic_targets(n, 61, 48)
        a = search_handle(w, image)
        a.target_buffer(64)
        a.append_targets(data)
        a.update_counts_buffer(96, 13, augment=True)
        out = a.training_batch(96, 13, augment=True)
        idx, sym = out["index"].cpu().numpy(), out["symmetry"].cpu().numpy()
        network.broadcast_novelty_set(a, None, 0)
        want = host_marked(n, kind, w, data["target_env"], idx, sym, bitset=image)
        assert (want != image).any()
        b = search_handle(w, want)
    else:
        a = search_handle(w)
        src = image
        if source == "pinned":
            src = capi.pinned_array((SET_BYTES,), np.uint8)
            src[:] = image
        network.broadcast_novelty_set(a, src, 0)
        a.sync()
        b = search_handle(w, image)
    assert np.array_equal(network.read_novelty_set(a), network.read_novelty_set(b))
    same_run(a, b, run(a, 4, 100), run(b, 4, 100))
    assert a.status() == 0
    a.close()
    b.close()
    if source == "pinned":
        capi.lib().tz_host_free(src.ctypes.data)


def test_swap_is_between_moves():
    w = hash_inputs(6, "simhash", 22)
    old, new = random_image(6), capi.pinned_array((SET_BYTES,), np.uint8)
    new[:] = random_image(7)
    # A: move, generation, move with no host synchronisation in between
    a = search_handle(w, old)
    a.selfplay_move(selfplay_params(200))
    network.broadcast_novelty_set(a, new, 0)
    a.selfplay_move(selfplay_params(201))
    roots_a = [a.root_children()]
    # B: the same with tz_set_simhash between the moves (which waits)
    b = search_handle(w, old)
    b.selfplay_move(selfplay_params(200))
    network.set_simhash(b, w, np.array(new))
    b.selfplay_move(selfplay_params(201))
    roots_b = [b.root_children()]
    same_run(a, b, roots_a, roots_b)
    a.close()
    b.close()
    capi.lib().tz_host_free(new.ctypes.data)


def test_generation_host_errors_change_nothing():
    w = hash_inputs(6, "simhash", 23)
    m = search_handle(w, random_image(8))
    before = network.read_novelty_set(m)
    rc = capi.lib().tz_broadcast_novelty_set(m.handle, None, 1)
    assert rc == EINVAL
    rc = capi.lib().tz_broadcast_novelty_set(m.handle, None, -1)
    assert rc == EINVAL
    assert np.array_equal(network.read_novelty_set(m), before)
    m.close()
    # the root needs a hash
    nohash = capi.BatchedMCTS(6, HK, 4, arena_slots=4096)
    network.set_weights(nohash, weights.random_init(6, seed=3, blocks=1))
    assert capi.lib().tz_broadcast_novelty_set(nohash.handle, None, 0) == ENOWEIGHTS
    nohash.close()


# ---- two ranks ---------------------------------------------------------------------------------------------------

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _digest(image):
    return hashlib.sha256(image.tobytes()).hexdigest()


def _worker(rank, world, port, out):
    import torch.distributed as dist

    from takzero_b200 import distributed as tzd

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n = 6
        w = hash_inputs(n, "simhash", 31)
        m = capi.BatchedMCTS(n, HK, 16, device=rank, arena_slots=4096)
        tzd.init_comm(m, rank, world)
        network.set_weights(m, weights.random_init(n, seed=3, blocks=1))
        network.set_simhash(m, w)
        data = synthetic_targets(n, 71, 64)
        states = data["target_env"]
        actions = [[] for _ in range(16)]
        if rank == 0:
            m.target_buffer(64)
            m.append_targets(data)
            m.update_counts_buffer(64, 9, augment=False)
        network.broadcast_novelty_set(m, None, 0)
        image = network.read_novelty_set(m)
        variances = [network.evaluate(m, states[i:i + 16], actions)[2] for i in range(0, 64, 16)]
        res = {"digest": _digest(image), "bits": int(np.unpackbits(image[image != 0]).sum()),
               "variances": np.concatenate(variances).view(np.uint32).tolist(), "status": m.status()}
        # a rank with the other hash kind: flagged, keeps its set; the root marks more and sends again
        if rank == 1:
            network.set_lcghash(m, hash_inputs(n, "lcghash", 32), image)
        else:
            m.update_counts_buffer(64, 10, augment=True)
        network.broadcast_novelty_set(m, None, 0)
        image2 = network.read_novelty_set(m)
        res.update(digest2=_digest(image2), status2=m.status())
        out[rank] = res
        m.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_share_the_roots_set():
    import torch.multiprocessing as mp

    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    r0, r1 = out[0], out[1]
    assert r0["bits"] > 0 and r0["digest"] == r1["digest"]
    assert r0["variances"] == r1["variances"]
    assert r0["status"] == 0 and r1["status"] == 0
    assert r0["status2"] == 0 and r0["digest2"] != r0["digest"]
    assert r1["status2"] == STATUS_WEIGHTS_MISMATCH and r1["digest2"] == r1["digest"]
