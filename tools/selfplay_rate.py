"""Cost of keeping resident self-play's training data, on the 6x6 headline configuration of bench.py (8192 games,
k = 16, 256 simulations, fp16, bench's weights).  One command alternates, `--rounds` times:
  (a) tz_selfplay_move without recording;
  (b) tz_selfplay_move with recording and a tz_selfplay_read after every move;
  (c) the `selfplay` binary without and with --resident, in moves per second of wall clock (process start, model load
      and the first move included, so compare the two with each other, not with (a) / (b)).
Prints one JSON object: simulations/s of (a) and (b), read time and bytes per move, the per-game high-water mark of
the record regions, the binary's rates, and the card's name and power limit read in the same run.

    python tools/selfplay_rate.py [--moves 6] [--rounds 3] [--games 8192] [--binary-moves 6] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench import ALLOWED_DROP, HALF_KOMI, SAMPLE_THRESHOLD, TARGET_BETA, WEIGHTED_RANDOM_PLIES, WORKLOADS, \
    target_visitations  # noqa: E402

# bytes of one queued target / policy entry / replay / replay move as tz_selfplay_read copies them
TARGET_BYTES, POLICY_BYTES, REPLAY_BYTES, MOVE_BYTES = 384 + 4 + 4 + 4 + 8 + 4, 2 + 4, 384 + 4 * 5 + 8 + 1, 2


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def timed_moves(m, sp, moves, read):
    m.sync()
    c0 = m.counters().simulations
    read_s, read_bytes, hw = 0.0, 0, 0
    t0 = time.perf_counter()
    for _ in range(moves):
        m.selfplay_move(sp)
        if read:
            m.sync()  # the read's own time only
            t = time.perf_counter()
            d = m.selfplay_read()
            read_s += time.perf_counter() - t
            read_bytes += (d["n_targets"] * TARGET_BYTES + d["n_policy"] * POLICY_BYTES +
                           d["n_replays"] * REPLAY_BYTES + d["n_moves"] * MOVE_BYTES)
            hw = max(hw, d["high_water_bytes"])
    m.sync()
    dt = time.perf_counter() - t0
    if m.status():
        raise SystemExit(f"device status 0x{m.status():x}")
    sims = m.counters().simulations - c0
    return {"sims_per_s": sims / dt, "seconds": dt, "read_ms_per_move": 1e3 * read_s / moves if read else None,
            "read_bytes_per_move": read_bytes / moves if read else None, "high_water_bytes": hw if read else None}


def binary_rate(exe, weights_path, args, resident):
    with tempfile.TemporaryDirectory() as d:
        cmd = [exe, "--directory", d, "--weights", weights_path, "--board", "6", "--half-komi", str(HALF_KOMI),
               "--games", str(args.games), "--sampled-actions", "16", "--budget", "256", "--moves",
               str(args.binary_moves), "--seed", "1"] + (["--resident"] if resident else [])
        t0 = time.perf_counter()
        out = subprocess.run(cmd, capture_output=True, text=True)
        dt = time.perf_counter() - t0
        if out.returncode != 0:
            raise SystemExit(out.stderr)
        size = sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))
    return {"moves_per_s": args.binary_moves / dt, "seconds": dt, "bytes_written": size}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--moves", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--games", type=int, default=WORKLOADS["6x6_selfplay"]["games"])
    ap.add_argument("--binary-moves", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    from takzero_b200 import build as tz_build
    from takzero_b200 import capi, network, weights

    tz_build.build()
    wl = WORKLOADS["6x6_selfplay"]
    k, budget = wl["k"], wl["budget"]
    w = weights.random_init(6, seed=123)  # bench.py's weights
    m = capi.BatchedMCTS(6, HALF_KOMI, args.games)
    network.set_weights(m, w, network.DTYPE_F16)
    m.set_agent(capi.AGENT_NETWORK)
    m.new_openings(seed=1)
    sp = capi.SelfplayParams(k, budget, 0.0, WEIGHTED_RANDOM_PLIES, SAMPLE_THRESHOLD, ALLOWED_DROP,
                             target_visitations(k, budget), TARGET_BETA, 1)
    for _ in range(args.warmup):
        m.selfplay_move(sp)
    exe = os.path.join(os.path.dirname(capi.LIB_PATH), "bin", "selfplay")
    res = {"card": card(), "games": args.games, "k": k, "budget": budget, "dtype": "fp16", "rounds": []}
    with tempfile.TemporaryDirectory() as wd:
        wpath = os.path.join(wd, "model.tzw")
        weights.save_tzw(wpath, w)
        for _ in range(args.rounds):
            r = {"a_off": timed_moves(m, sp, args.moves, False)}
            m.selfplay_record(True)
            r["b_record_read"] = timed_moves(m, sp, args.moves, True)
            m.selfplay_record(False)
            r["c_binary_host"] = binary_rate(exe, wpath, args, False)
            r["c_binary_resident"] = binary_rate(exe, wpath, args, True)
            res["rounds"].append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
    m.close()
    rounds = res["rounds"]
    a = sum(r["a_off"]["sims_per_s"] for r in rounds) / len(rounds)
    b = sum(r["b_record_read"]["sims_per_s"] for r in rounds) / len(rounds)
    res["summary"] = {
        "a_sims_per_s": a, "b_sims_per_s": b, "b_over_a": b / a,
        "read_ms_per_move": sum(r["b_record_read"]["read_ms_per_move"] for r in rounds) / len(rounds),
        "read_bytes_per_move": sum(r["b_record_read"]["read_bytes_per_move"] for r in rounds) / len(rounds),
        "high_water_bytes_per_game": max(r["b_record_read"]["high_water_bytes"] for r in rounds),
        "binary_host_moves_per_s": sum(r["c_binary_host"]["moves_per_s"] for r in rounds) / len(rounds),
        "binary_resident_moves_per_s": sum(r["c_binary_resident"]["moves_per_s"] for r in rounds) / len(rounds),
    }
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
