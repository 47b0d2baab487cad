"""Host-side mirror of the reference's `Network` / `Agent` surface for the device ResNet
(takzero/src/network/mod.rs:10-45, net6_simhash.rs:259-324): weight upload and the
evaluate / encode hooks of the C ABI.  All math happens in libtakzero_b200.so."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Sequence

import numpy as np

from . import capi


class _Tensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.POINTER(C.c_float)), ("shape", C.POINTER(C.c_int64)),
                ("ndim", C.c_int)]


_MODEL_TENSOR_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_float), C.POINTER(C.c_int64),
                               C.c_int)

_declared = False


def _declare():
    global _declared
    if _declared:
        return
    vp, i32 = C.c_void_p, C.c_int
    capi.declare("tz_set_weights", [vp, C.POINTER(_Tensor), i32], i32)
    capi.declare("tz_evaluate", [vp, vp, i32, vp, vp, i32, vp, vp, vp], i32)
    capi.declare("tz_encode_planes", [vp, vp, i32, vp], i32)
    capi.declare("tz_set_network_dtype", [vp, i32], i32)
    capi.declare("tz_set_simhash", [vp, vp, vp], i32)
    capi.declare("tz_simhash_indices", [vp, vp, i32, vp], i32)
    capi.declare("tz_set_lcghash", [vp, vp, vp], i32)
    capi.declare("tz_lcghash_indices", [vp, vp, i32, vp], i32)
    capi.declare("tz_update_counts", [vp, vp, i32], i32)
    capi.declare("tz_read_novelty_set", [vp, vp, C.c_size_t], i32)
    capi.declare("tz_debug_layer_limit", [vp, i32], i32)
    capi.declare("tz_debug_activations", [vp, i32, i32, vp], i32)
    capi.declare("tz_debug_time_tower", [vp, i32, i32, C.POINTER(C.c_double)], i32)
    capi.declare("tz_load_model", [vp, C.c_char_p], i32)
    capi.declare("tz_load_model_ex", [vp, C.c_char_p, i32], i32)
    capi.declare("tz_debug_network_mode", [vp, i32, i32, i32], i32)
    capi.declare("tz_debug_weight_set", [vp, vp, C.c_size_t, C.POINTER(C.c_size_t)], i32)
    capi.declare("tz_debug_expf", [vp, vp, i32, vp], i32)
    capi.declare("tz_comm_unique_id", [vp], i32)
    capi.declare("tz_comm_init", [vp, vp, i32, i32], i32)
    capi.declare("tz_comm_destroy", [vp], i32)
    capi.declare("tz_broadcast_weights", [vp, C.POINTER(_Tensor), i32, i32, i32], i32)
    capi.declare("tz_broadcast_novelty_set", [vp, vp, i32], i32)
    capi.declare("tz_weight_generation", [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_double)], i32)
    capi.declare("tz_allreduce_sum", [vp, vp, i32], i32)
    capi.declare("tz_read_model_file", [C.c_char_p, _MODEL_TENSOR_FN, vp], i32)
    _declared = True


DTYPE_BF16, DTYPE_F16 = 0, 1
DTYPE_DEFAULT = DTYPE_F16  # the library's default: the mode that meets the >= 99 % chosen-move agreement bar


def _tensor_array(tensors: Dict[str, np.ndarray]):
    keep = []
    arr = (_Tensor * len(tensors))()
    for i, (name, t) in enumerate(tensors.items()):
        a = np.ascontiguousarray(t, dtype=np.float32)
        shape = (C.c_int64 * a.ndim)(*a.shape)
        keep += [a, shape]
        arr[i] = _Tensor(name.encode(), a.ctypes.data_as(C.POINTER(C.c_float)), shape, a.ndim)
    return arr, keep


def set_weights(mcts: capi.BatchedMCTS, tensors: Dict[str, np.ndarray], dtype: int = DTYPE_DEFAULT) -> None:
    """`Net::load`: upload named f32 tensors (PyTorch layout, names in include/takzero_b200.h); `dtype` is the
    16-bit type of weights and activations on the device (fp16 by default).  The tensors are staged by the library
    before the call returns; BatchNorm folding and the weight arrangement run on the GPU beside the search."""
    _declare()
    capi._check(capi.lib().tz_set_network_dtype(mcts.handle, dtype))
    arr, _keep = _tensor_array(tensors)
    capi._check(capi.lib().tz_set_weights(mcts.handle, arr, len(tensors)))


def broadcast_weights(mcts: capi.BatchedMCTS, tensors: Dict[str, np.ndarray] | None, root: int = 0,
                      res_blocks: int = 0, dtype: int = DTYPE_DEFAULT) -> None:
    """One weight generation on every rank of the handle's communicator (`tz_broadcast_weights`, collective): the
    root passes the tensors, the others None; also valid without a communicator (= set_weights).  The RND estimator
    of a 5x5 model (`rnd_learning.*`, `rnd_target.*`, `min`, `max`) is not broadcast: the root takes it as set_weights
    does, and the other ranks keep the one they had."""
    _declare()
    capi._check(capi.lib().tz_set_network_dtype(mcts.handle, dtype))
    if tensors is None:
        capi._check(capi.lib().tz_broadcast_weights(mcts.handle, None, 0, res_blocks, root))
    else:
        arr, _keep = _tensor_array(tensors)
        capi._check(capi.lib().tz_broadcast_weights(mcts.handle, arr, len(tensors), res_blocks, root))


def broadcast_novelty_set(mcts: capi.BatchedMCTS, bitset: np.ndarray | None = None, root: int = 0) -> None:
    """One novelty-set generation on every rank of the handle's communicator (`tz_broadcast_novelty_set`,
    collective): the root passes a `bitvec.bin` image (2^29 uint8; from capi.pinned_array it is uploaded in place and
    must stay unchanged until mcts.sync()) or None for its own current set; the other ranks pass None.  Every rank
    swaps to the new set for the launches it enqueues afterwards."""
    _declare()
    b = None
    if bitset is not None:
        b = np.ascontiguousarray(bitset, dtype=np.uint8)
        assert b.size == 1 << 29
    capi._check(capi.lib().tz_broadcast_novelty_set(mcts.handle, capi._ptr(b), root))


def weight_generation(mcts: capi.BatchedMCTS):
    """(generations so far, device milliseconds of the last one: upload + fold + broadcast)."""
    _declare()
    gen, ms = C.c_uint64(), C.c_double()
    capi._check(capi.lib().tz_weight_generation(mcts.handle, C.byref(gen), C.byref(ms)))
    return gen.value, ms.value


def comm_unique_id() -> bytes:
    _declare()
    buf = C.create_string_buffer(128)
    capi._check(capi.lib().tz_comm_unique_id(buf))
    return buf.raw


def comm_init(mcts: capi.BatchedMCTS, unique_id: bytes | None, nranks: int, rank: int) -> None:
    _declare()
    capi._check(capi.lib().tz_comm_init(mcts.handle, unique_id, nranks, rank))


def allreduce_sum(mcts: capi.BatchedMCTS, values) -> list:
    """Whole-job totals of per-rank counters over the handle's communicator (ncclAllReduce)."""
    _declare()
    a = np.ascontiguousarray(values, dtype=np.uint64)
    capi._check(capi.lib().tz_allreduce_sum(mcts.handle, capi._ptr(a), len(a)))
    return [int(x) for x in a]


def debug_network_mode(mcts: capi.BatchedMCTS, per_layer_launches: bool = False, chunk_min_tiles: int = -1,
                       drop_progress: bool = False) -> None:
    """Test / measurement hook (`tz_debug_network_mode`): launch structure for the NEXT set_weights, watchdog test."""
    _declare()
    capi._check(capi.lib().tz_debug_network_mode(mcts.handle, int(per_layer_launches), chunk_min_tiles,
                                                 int(drop_progress)))


def weight_set(mcts: capi.BatchedMCTS) -> np.ndarray:
    """The active weight set as bytes (parity hook for the on-device folding / arrangement)."""
    _declare()
    size = C.c_size_t()
    capi._check(capi.lib().tz_debug_weight_set(mcts.handle, None, 0, C.byref(size)))
    out = np.zeros(size.value, dtype=np.uint8)
    capi._check(capi.lib().tz_debug_weight_set(mcts.handle, capi._ptr(out), out.size, C.byref(size)))
    return out


def load_model(mcts: capi.BatchedMCTS, path: str, dtype: int = DTYPE_DEFAULT, allow_missing_set: bool = False) -> None:
    """`Net::load(path, device)` (network/mod.rs:20-27, net6_simhash.rs:164-181): read the reference's
    `model_latest.ot` (tch VarStore archive; also a `torch.save` state dict or a TZW1 file) inside the library,
    upload it, and take the SimHash matrix / `bitvec.bin` sidecar when the file has them (a missing sidecar is an
    error like in the reference unless `allow_missing_set`)."""
    _declare()
    capi._check(capi.lib().tz_set_network_dtype(mcts.handle, dtype))
    capi._check(capi.lib().tz_load_model_ex(mcts.handle, str(path).encode(), int(allow_missing_set)))


def read_model_file(path: str, stored_names: bool = False) -> Dict[str, np.ndarray]:
    """`Tensor::load_multi`: every tensor of a model file as f32, keyed by the library's tensor names (or by the
    names stored in the file).  Parsed by the C++ reader of the library; needs no GPU."""
    _declare()
    out: Dict[str, np.ndarray] = {}

    def cb(_ctx, name, stored, data, shape, ndim):
        shp = tuple(shape[i] for i in range(ndim))
        n = int(np.prod(shp)) if ndim else 1
        a = np.ctypeslib.as_array(data, shape=(n,)).copy() if n else np.zeros(0, np.float32)
        out[(stored if stored_names else name).decode()] = a.reshape(shp)

    capi._check(capi.lib().tz_read_model_file(str(path).encode(), _MODEL_TENSOR_FN(cb), None))
    return out


def evaluate(mcts: capi.BatchedMCTS, states: np.ndarray, actions: Sequence[Sequence[int]]):
    """`Agent::policy_value_uncertainty` for host positions: (logits list, values, variances)."""
    _declare()
    states = np.ascontiguousarray(states, dtype=capi.STATE_DTYPE)
    count, M = len(states), mcts.move_stride
    act = np.zeros((count, M), dtype=np.uint16)
    nact = np.zeros(count, dtype=np.int32)
    for i, a in enumerate(actions):
        act[i, : len(a)] = a
        nact[i] = len(a)
    logits = np.zeros((count, M), dtype=np.float32)
    values = np.zeros(count, dtype=np.float32)
    variances = np.zeros(count, dtype=np.float32)
    p = capi._ptr
    capi._check(capi.lib().tz_evaluate(mcts.handle, p(states), count, p(act), p(nact), M, p(logits), p(values),
                                       p(variances)))
    return [logits[i, : nact[i]].copy() for i in range(count)], values, variances


def encode_planes(mcts: capi.BatchedMCTS, states: np.ndarray) -> np.ndarray:
    """`game_repr` (network/repr.rs:169-228): f32 [count, C, N, N]."""
    _declare()
    states = np.ascontiguousarray(states, dtype=capi.STATE_DTYPE)
    out = np.zeros((len(states), mcts.input_channels, mcts.n, mcts.n), dtype=np.float32)
    capi._check(capi.lib().tz_encode_planes(mcts.handle, capi._ptr(states), len(states), capi._ptr(out)))
    return out


def debug_layer_limit(mcts: capi.BatchedMCTS, limit: int) -> None:
    _declare()
    capi._check(capi.lib().tz_debug_layer_limit(mcts.handle, limit))


def debug_activations(mcts: capi.BatchedMCTS, which: int, count: int) -> np.ndarray:
    _declare()
    ch = 64 if which == 2 else 256
    out = np.zeros((count, mcts.n * mcts.n, ch), dtype=np.float32)
    capi._check(capi.lib().tz_debug_activations(mcts.handle, which, count, capi._ptr(out)))
    return out


def time_tower(mcts: capi.BatchedMCTS, count: int, reps: int = 20) -> float:
    """Mean milliseconds per tower-convolution launch over `count` positions (tuning hook)."""
    _declare()
    ms = C.c_double()
    capi._check(capi.lib().tz_debug_time_tower(mcts.handle, count, reps, C.byref(ms)))
    return ms.value


def set_simhash(mcts: capi.BatchedMCTS, matrix: np.ndarray, bitset: np.ndarray | None = None) -> None:
    """SimHash matrix [C*N*N, 32] and optionally the 2^32-bit set as 2^29 bytes (`bitvec.bin`)."""
    _declare()
    m = np.ascontiguousarray(matrix, dtype=np.float32)
    assert m.shape == (mcts.input_channels * mcts.n * mcts.n, 32)
    b = None
    if bitset is not None:
        b = np.ascontiguousarray(bitset, dtype=np.uint8)
        assert b.size == 1 << 29
    capi._check(capi.lib().tz_set_simhash(mcts.handle, capi._ptr(m), capi._ptr(b)))


def simhash_indices(mcts: capi.BatchedMCTS, states: np.ndarray) -> np.ndarray:
    _declare()
    states = np.ascontiguousarray(states, dtype=capi.STATE_DTYPE)
    out = np.zeros(len(states), dtype=np.uint32)
    capi._check(capi.lib().tz_simhash_indices(mcts.handle, capi._ptr(states), len(states), capi._ptr(out)))
    return out


def set_lcghash(mcts: capi.BatchedMCTS, init: np.ndarray, bitset: np.ndarray | None = None) -> None:
    """LCG-hash novelty (net4_lcghash.rs): `lcghash_init` [C, N, N] and optionally the 2^32-bit set."""
    _declare()
    a = np.ascontiguousarray(init, dtype=np.float32)
    assert a.shape == (mcts.input_channels, mcts.n, mcts.n)
    b = None
    if bitset is not None:
        b = np.ascontiguousarray(bitset, dtype=np.uint8)
        assert b.size == 1 << 29
    capi._check(capi.lib().tz_set_lcghash(mcts.handle, capi._ptr(a), capi._ptr(b)))


def lcghash_indices(mcts: capi.BatchedMCTS, states: np.ndarray) -> np.ndarray:
    _declare()
    states = np.ascontiguousarray(states, dtype=capi.STATE_DTYPE)
    out = np.zeros(len(states), dtype=np.uint32)
    capi._check(capi.lib().tz_lcghash_indices(mcts.handle, capi._ptr(states), len(states), capi._ptr(out)))
    return out


def update_counts(mcts: capi.BatchedMCTS, states: np.ndarray) -> None:
    """`Net::update_counts` (net6_simhash.rs:236-241): mark these positions as seen in the novelty set."""
    _declare()
    states = np.ascontiguousarray(states, dtype=capi.STATE_DTYPE)
    capi._check(capi.lib().tz_update_counts(mcts.handle, capi._ptr(states), len(states)))


def read_novelty_set(mcts: capi.BatchedMCTS) -> np.ndarray:
    """The 2^29-byte image of the set, as the reference's `bitvec.bin` holds it."""
    _declare()
    out = np.empty(1 << 29, dtype=np.uint8)
    capi._check(capi.lib().tz_read_novelty_set(mcts.handle, capi._ptr(out), out.size))
    return out
