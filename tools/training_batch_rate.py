"""Rate of tz_training_batch on 6x6: a target buffer of 10^6 synthetic targets (about 6.5 GB, far larger than the
126 MB L2), drawn batches of 256 / 1024 / 4096 examples with augmentation, every output written (planes, policy,
mask, value, ube, index, symmetry).

The targets are seeded random playout positions (the oracle's rules) with random probabilities over their legal
moves; the positions repeat every --positions targets, the probabilities do not, and every target has its own slot.
For every batch size, after --warmup batches:
  - kernel time (`kernel_ms_profiler`): k_training_batch's mean device time over --calls launches, from
    torch.profiler's CUDA activity records.  tz_training_batch waits for the stream before it enqueues the kernel, so
    CUDA events around a run of calls would also time the host round trip between kernels; the activity records
    time the kernel alone;
  - call time (`call_ms_wall`): wall clock of --calls consecutive training_batch calls, each waiting for its result,
    as a learner calling it from Python sees it;
  - examples/s of both, and the bytes the kernel has to move (outputs written + slots read, from the shapes and the
    mean entry count) over the kernel time (`kernel_gbps`), also as a fraction of HBM_GBPS.
Prints one JSON object with the card's name and power limit read in the same run.

    python tools/training_batch_rate.py [--targets 1000000] [--calls 50] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

# HBM bandwidth a copy kernel measured on one B200 at a 1000 W power limit (GB/s): the bound this kernel works against
HBM_GBPS = 6543.4
N, HALF_KOMI = 6, 4


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def fill(m, targets, positions, seed):
    from oracle import oracle as O
    from takzero_b200 import capi

    pp = O.playout_positions(N, HALF_KOMI, seed, 4, positions)
    counts = pp["n_moves"].astype(np.int32)
    moves = np.concatenate([pp["moves"][i, :counts[i]] for i in range(positions)]).astype(np.uint16)
    offset = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.uint64)
    env = pp["states"].view(capi.STATE_DTYPE).reshape(positions)
    rng = np.random.default_rng(seed)
    keep = counts > 0
    for start in range(0, targets, positions):
        c = min(positions, targets - start)
        raw = rng.random(len(moves)).astype(np.float32) + np.float32(1e-6)
        sums = np.add.reduceat(raw, offset[keep].astype(np.int64))
        norm = np.zeros(positions, np.float32)
        norm[keep] = sums
        probs = raw / np.repeat(np.where(norm > 0, norm, 1), counts)
        m.append_targets({"target_env": env[:c], "target_value": rng.uniform(-1, 1, c).astype(np.float32),
                          "target_ube": rng.uniform(0, 4, c).astype(np.float32), "target_n": counts[:c],
                          "target_offset": offset[:c], "policy_moves": moves, "policy_probs": probs})
    return float(counts.mean())


def kernel_ms(m, batch, out, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(reps):
            m.training_batch(batch, 1000 + i, out=out)
    for e in prof.key_averages():
        if "k_training_batch" in e.key:
            total = getattr(e, "device_time_total", None)
            if total is None:
                total = e.cuda_time_total
            return total / e.count / 1e3
    raise SystemExit("k_training_batch not found in the profile")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--targets", type=int, default=1_000_000)
    ap.add_argument("--positions", type=int, default=20_000)
    ap.add_argument("--batches", default="256,1024,4096")
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    from takzero_b200 import build as tz_build
    from takzero_b200 import capi

    tz_build.build()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measures the B200")
    m = capi.BatchedMCTS(N, HALF_KOMI, 1)
    m.target_buffer(args.targets)
    t0 = time.perf_counter()
    mean_n = fill(m, args.targets, args.positions, seed=1)
    fill_s = time.perf_counter() - t0
    size, appended = m.target_buffer_info()
    nn, C, OC = N * N, m.input_channels, m.output_channels
    res = {"card": card(), "board": N, "targets": size, "appended": appended, "mean_entries": mean_n,
           "buffer_bytes": size * (384 + 12 + 6 * m.move_stride), "append_seconds": fill_s, "hbm_gbps": HBM_GBPS,
           "batches": []}
    for batch in (int(b) for b in args.batches.split(",")):
        shapes = m.training_shapes(batch)
        out = {k: torch.empty(s, dtype=getattr(torch, dt), device="cuda") for k, (s, dt) in shapes.items()}
        for i in range(args.warmup):
            m.training_batch(batch, i, out=out)
        t0 = time.perf_counter()
        for i in range(args.calls):
            m.training_batch(batch, 100 + i, out=out)
        call_s = (time.perf_counter() - t0) / args.calls
        k_ms = kernel_ms(m, batch, out, args.calls)
        written = batch * (4 * C * nn + 4 * OC * nn + OC * nn + 4 * 4)
        read = batch * (384 + 12 + 6 * mean_n)
        gbps = (written + read) / (k_ms * 1e-3) / 1e9
        r = {"batch": batch, "kernel_ms_profiler": k_ms, "kernel_examples_per_s": batch / (k_ms * 1e-3),
             "call_ms_wall": call_s * 1e3, "call_examples_per_s": batch / call_s, "bytes_written": written,
             "bytes_read": read, "kernel_gbps": gbps, "kernel_fraction_of_hbm": gbps / HBM_GBPS}
        res["batches"].append(r)
        print(json.dumps(r), file=sys.stderr, flush=True)
    m.close()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
