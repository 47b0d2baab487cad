"""Cost of the novelty set as part of a generation (tz_broadcast_novelty_set, tz_update_counts_buffer), in one command
on one B200 (the two-rank broadcast only where a second GPU is visible):
  - set generation (`generation_ms`): host clock around tz_broadcast_novelty_set + tz_sync on an idle 6x6 handle with a
    SimHash hash, for a pinned host image, a pageable host image and the handle's own set (NULL); --reps each;
  - the same broadcast from rank 0 to rank 1 over NCCL, on two GPUs;
  - k_mark_batch (`kernel_ms_profiler`): mean device time of tz_update_counts_buffer at --batches examples with
    augmentation, on a 6x6 target buffer of --targets synthetic targets, from torch.profiler's CUDA activity records;
  - self-play on bench.py's 6x6 headline configuration (8192 games, k = 16, 256 simulations, fp16): simulations/s
    with a weight generation before every move (a) against a weight generation plus a set generation from a pinned
    image before every move (b), alternated over --rounds rounds of --moves moves.
Prints one JSON object with the card's name and power limit read in the same run.

    python tools/novelty_generation_rate.py [--reps 5] [--targets 1000000] [--moves 4] [--rounds 3] [--out FILE]"""
import argparse
import json
import os
import socket
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench import ALLOWED_DROP, HALF_KOMI, SAMPLE_THRESHOLD, TARGET_BETA, WEIGHTED_RANDOM_PLIES, WORKLOADS, \
    target_visitations  # noqa: E402
from training_batch_rate import card, fill  # noqa: E402

SET_BYTES = 1 << 29
N = 6


def simhash_matrix(seed):
    cin = 2 * (2 * N + 5) + 2
    return np.random.default_rng(seed).standard_normal((cin * N * N, 32)).astype(np.float32)


def image(seed):
    return np.random.default_rng(seed).integers(0, 256, SET_BYTES, dtype=np.uint8)


def generation_ms(m, src, reps):
    from takzero_b200 import network

    out = []
    for _ in range(reps + 1):  # the first one allocates the second set (and the staging of a pageable image)
        m.sync()
        t0 = time.perf_counter()
        network.broadcast_novelty_set(m, src, 0)
        m.sync()
        out.append((time.perf_counter() - t0) * 1e3)
    return {"ms_each": out[1:], "ms_mean": float(np.mean(out[1:])), "first_call_ms": out[0]}


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _rank(rank, world, port, reps, out):
    import torch.distributed as dist

    from takzero_b200 import capi, network, weights
    from takzero_b200 import distributed as tzd

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        m = capi.BatchedMCTS(N, HALF_KOMI, 64, device=rank, arena_slots=4096)
        tzd.init_comm(m, rank, world)
        network.set_weights(m, weights.random_init(N, seed=3, blocks=1))
        network.set_simhash(m, simhash_matrix(1))
        times = []
        for _ in range(reps + 1):
            m.sync()
            dist.barrier()
            t0 = time.perf_counter()
            network.broadcast_novelty_set(m, None, 0)
            m.sync()
            times.append((time.perf_counter() - t0) * 1e3)
        out[rank] = {"ms_each": times[1:], "ms_mean": float(np.mean(times[1:])), "status": m.status()}
        m.close()
    finally:
        dist.destroy_process_group()


def two_rank_broadcast(reps):
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 2:
        return "not measured: one GPU visible"
    out = mp.Manager().dict()
    mp.spawn(_rank, args=(2, _free_port(), reps, out), nprocs=2, join=True)
    return {"rank0": dict(out[0]), "rank1": dict(out[1])}


def mark_kernel_ms(m, batch, reps):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(reps):
            m.update_counts_buffer(batch, 1000 + i, augment=True)
        m.sync()
    for e in prof.key_averages():
        if "k_mark_batch" in e.key:
            total = getattr(e, "device_time_total", None)
            if total is None:
                total = e.cuda_time_total
            return total / e.count / 1e3
    raise SystemExit("k_mark_batch not found in the profile")


def timed_moves(m, sp, moves, generation):
    m.sync()
    c0 = m.counters().simulations
    t0 = time.perf_counter()
    for _ in range(moves):
        generation()
        m.selfplay_move(sp)
    m.sync()
    dt = time.perf_counter() - t0
    if m.status():
        raise SystemExit(f"device status 0x{m.status():x}")
    return {"sims_per_s": (m.counters().simulations - c0) / dt, "seconds": dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--targets", type=int, default=1_000_000)
    ap.add_argument("--positions", type=int, default=20_000)
    ap.add_argument("--batches", default="256,1024,4096")
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--games", type=int, default=WORKLOADS["6x6_selfplay"]["games"])
    ap.add_argument("--moves", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    from takzero_b200 import build as tz_build
    from takzero_b200 import capi, network, weights

    tz_build.build()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measures the B200")
    res = {"card": card(), "board": N, "set_bytes": SET_BYTES}

    # set generations on an idle handle
    m = capi.BatchedMCTS(N, HALF_KOMI, 64, arena_slots=4096)
    network.set_weights(m, weights.random_init(N, seed=3, blocks=1))
    network.set_simhash(m, simhash_matrix(1), image(2))
    pinned = capi.pinned_array((SET_BYTES,), np.uint8)
    pinned[:] = image(3)
    pageable = image(4)
    res["generation"] = {"pinned": generation_ms(m, pinned, args.reps),
                         "pageable": generation_ms(m, pageable, args.reps),
                         "own_set_null": generation_ms(m, None, args.reps)}
    print(json.dumps(res["generation"]), file=sys.stderr, flush=True)

    # marking kernel on a large buffer
    m.target_buffer(args.targets)
    fill(m, args.targets, args.positions, seed=1)
    res["targets"] = m.target_buffer_info()[0]
    res["mark"] = []
    for batch in (int(b) for b in args.batches.split(",")):
        for i in range(5):
            m.update_counts_buffer(batch, i, augment=True)
        m.sync()
        k_ms = mark_kernel_ms(m, batch, args.calls)
        r = {"batch": batch, "kernel_ms_profiler": k_ms, "examples_per_s": batch / (k_ms * 1e-3)}
        res["mark"].append(r)
        print(json.dumps(r), file=sys.stderr, flush=True)
    m.close()

    res["broadcast_2gpu"] = two_rank_broadcast(args.reps)

    # self-play with a weight generation per move, with and without a set generation
    wl = WORKLOADS["6x6_selfplay"]
    k, budget = wl["k"], wl["budget"]
    w = weights.random_init(N, seed=123)  # bench.py's weights
    m = capi.BatchedMCTS(N, HALF_KOMI, args.games)
    network.set_weights(m, w, network.DTYPE_F16)
    network.set_simhash(m, simhash_matrix(1), image(2))
    m.set_agent(capi.AGENT_NETWORK)
    m.new_openings(seed=1)
    sp = capi.SelfplayParams(k, budget, 0.0, WEIGHTED_RANDOM_PLIES, SAMPLE_THRESHOLD, ALLOWED_DROP,
                             target_visitations(k, budget), TARGET_BETA, 1)
    weights_only = lambda: network.broadcast_weights(m, w, root=0)
    with_set = lambda: (network.broadcast_weights(m, w, root=0), network.broadcast_novelty_set(m, pinned, 0))
    for _ in range(args.warmup):
        with_set()
        m.selfplay_move(sp)
    rounds = []
    for _ in range(args.rounds):
        r = {"a_weights": timed_moves(m, sp, args.moves, weights_only),
             "b_weights_and_set": timed_moves(m, sp, args.moves, with_set)}
        rounds.append(r)
        print(json.dumps(r), file=sys.stderr, flush=True)
    m.close()
    capi.lib().tz_host_free(pinned.ctypes.data)
    a = [r["a_weights"]["sims_per_s"] for r in rounds]
    b = [r["b_weights_and_set"]["sims_per_s"] for r in rounds]
    res["selfplay"] = {"games": args.games, "k": k, "budget": budget, "dtype": "fp16", "moves_per_leg": args.moves,
                       "rounds": rounds, "a_sims_per_s": float(np.mean(a)), "b_sims_per_s": float(np.mean(b)),
                       "b_over_a": float(np.mean(b) / np.mean(a)), "a_spread": [min(a), max(a)],
                       "b_spread": [min(b), max(b)]}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
