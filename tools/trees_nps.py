"""Many single trees at once (tz_trees_simulate_batch): aggregate search speed against the number of trees.
6x6, bench.py's seeded random weights (weights.random_init(6, seed=123)), fp16, 128 leaves per tree and batch (tei's
batch), T trees from seeded openings.  For each T: nodes/s over all trees (counters().simulations over a synchronised
wall clock), ms per batch (one batch = every tree's simulate_batch and one network pass) and network positions per batch.

--baseline DIR also times the one-tree path (tools/tei_nps.py 6 128 <batches>) of this tree and of another checkout DIR
(built), alternating, --rounds times each, in fresh processes; the spread of each side's rounds is the run-to-run noise.

    python tools/trees_nps.py [--trees 1,4,16,64] [--batches 100] [--baseline DIR] [--rounds 3]"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def trees_rate(T, batches, warmup, w):
    from takzero_b200 import capi, network

    batch = 128
    m = capi.BatchedMCTS(6, 4, T, tree_batch=T * batch, arena_slots=1 << 22)
    network.set_weights(m, w, network.DTYPE_F16)
    m.set_agent(capi.AGENT_NETWORK)
    m.new_openings(seed=1)
    for _ in range(warmup):
        m.trees_simulate_batch(0.0, batch)
    m.sync()
    c0 = m.counters()
    t0 = time.perf_counter()
    for _ in range(batches):
        m.trees_simulate_batch(0.0, batch)
    m.sync()
    dt = time.perf_counter() - t0
    c1 = m.counters()
    if m.status():
        raise SystemExit(f"device status 0x{m.status():x}")
    m.close()
    sims = c1.simulations - c0.simulations
    return {"trees": T, "nodes_per_s": sims / dt, "ms_per_batch": dt / batches * 1e3,
            "positions_per_batch": (c1.evaluations - c0.evaluations) / batches}


def tei_nps(root, batches):
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "tei_nps.py"), "6", "128", str(batches)],
                         capture_output=True, text=True, cwd=root)
    if out.returncode != 0:
        raise SystemExit(out.stderr)
    line = out.stdout.strip().splitlines()[-1]
    return float(line.split(": ")[1].split(" nodes/s")[0].replace(",", "")), line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", default="1,4,16,64")
    ap.add_argument("--batches", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--baseline", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()

    from takzero_b200 import build as tz_build
    from takzero_b200 import weights

    tz_build.build()
    print(f"card, power limit: {card()}", flush=True)
    print("6x6, fp16, bench's random weights, 128 leaves per tree and batch", flush=True)
    w = weights.random_init(6, seed=123)
    base = None
    for T in (int(t) for t in args.trees.split(",")):
        r = trees_rate(T, args.batches, args.warmup, w)
        if base is None:
            base = r["nodes_per_s"] / T
        print(f"  T = {T:3d}: {r['nodes_per_s']:>12,.0f} nodes/s  {r['ms_per_batch']:7.2f} ms per batch  "
              f"{r['positions_per_batch']:7.1f} network positions per batch  "
              f"({r['nodes_per_s'] / base:5.2f}x the first T's rate per tree)", flush=True)
    if args.baseline:
        print(f"one-tree path, tools/tei_nps.py 6 128 {args.batches}, alternating, {args.rounds} rounds:", flush=True)
        here, there = [], []
        for _ in range(args.rounds):
            for side, root, acc in (("this tree", ROOT, here), ("baseline", os.path.abspath(args.baseline), there)):
                rate, line = tei_nps(root, args.batches)
                acc.append(rate)
                print(f"  {side:9s} {line}", flush=True)
        for side, acc in (("this tree", here), ("baseline", there)):
            print(f"  {side:9s} mean {sum(acc) / len(acc):,.0f} nodes/s, min {min(acc):,.0f}, max {max(acc):,.0f}")
        print(f"  this tree / baseline: {sum(here) / sum(there):.4f}")


if __name__ == "__main__":
    main()
