#!/usr/bin/env python
"""bench.py -- self-play MCTS simulations/s (and positions/s) of the batched self-play search.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME]      our arm (CUDA library)
  python bench.py --impl reference [...]                                     restated reference on the host cores

Workloads (BASELINE.json `configs`):
  6x6_selfplay (default)  configs[2] / configs[3]: 6x6 Tak, half komi 4, 8192 concurrent games per GPU, k = 16 sampled
                          actions, 256 simulations/move, random-init 16x256 ResNet (torch seed 123)
  4x4_1024                configs[1]: 4x4 Tak, 1024 concurrent games, k = 16, 128 simulations/move, 16x256 ResNet
  5x5_selfplay            (not a BASELINE config; the third board size of the north star) 5x5, 8192 games, 20x256 ResNet
  reanalyze_1m            configs[4]: 6x6 `reanalyze` fresh-target search over a synthetic replay buffer of 1 M positions
                          (all plies of random playouts), positions sharded over the GPUs by contiguous index range,
                          batches of 8192 fresh roots per GPU, k = 16, 256 simulations

A self-play "step" is one move of every concurrent game: the model reload of selfplay/src/main.rs:107 (a weight
GENERATION: upload + fold on the GPU, NCCL broadcast from rank 0 for N > 1, set swap), Gumbel sequential halving
(1 + budget lock-step simulations), targets, action selection, step, restart (search/node/batched.rs:207-409,
selfplay/src/main.rs:138-153,238-329).  A reanalyze step is one batch (reanalyze/src/main.rs:147-235).  Every rank runs
its own games (weak scaling); there is no collective inside a simulation.

`value`  : simulations/s with everything resident in HBM (tz_selfplay_move / tz_reanalyze_batch, no per-step host
           buffers except the weight generation's tensors on rank 0), Gumbel noise drawn by the library.
`e2e`    : the same loop through the host-buffer C ABI: Gumbel noise INJECTED from pinned host memory, moves /
           improved-policy targets / terminals read back every step (so the two legs use different noise sources).
`roofline`: the fused network kernel (tcgen05), sampled with CUDA events inside the timed region.
`cpu_baseline`: the restated reference (oracle C search + libtorch-CPU f32 forward, 128 games in lock-step like
           selfplay/src/main.rs:37) on this box's host cores, bounded sample.

--dump-outputs DIR writes what the last timed step of the `value` leg computed as DIR/<name>.npy (float32, float64 for
integers wider than 16 bits, so every value is exact), rank 0's games only, for comparing two builds output for output: after a
self-play move the games' new positions and the children of their new roots (the subtree the search grew), after a
reanalyze batch the targets tz_reanalyze_read returns.  Per-game arrays keep a fixed, seeded sample of DUMP_GAMES games
(`games.npy` lists them); the inputs are seeded, so the same arguments give the same inputs on every run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HALF_KOMI = 4
WEIGHTED_RANDOM_PLIES, SAMPLE_THRESHOLD, ALLOWED_DROP, TARGET_BETA = 10, 32, 0.5, 0.25
CPU_GAMES = 128  # BATCH_SIZE of the reference process (selfplay/src/main.rs:37)
UNIT = "simulations/s"

WORKLOADS = {
    "6x6_selfplay": dict(kind="selfplay", n=6, games=int(os.environ.get("TZ_BENCH_GAMES", "8192")), k=16, budget=256,
                         metric="self-play MCTS simulations/sec, 6x6 Tak"),
    "4x4_1024": dict(kind="selfplay", n=4, games=1024, k=16, budget=128,
                     metric="self-play MCTS simulations/sec, 4x4 Tak"),
    "5x5_selfplay": dict(kind="selfplay", n=5, games=8192, k=16, budget=256,
                         metric="self-play MCTS simulations/sec, 5x5 Tak"),
    "reanalyze_1m": dict(kind="reanalyze", n=6, games=8192, k=16, budget=256, buffer=1_000_000,
                         metric="reanalyze MCTS simulations/sec, 6x6 Tak"),
}


def target_visitations(k: int, budget: int) -> float:
    # IMPROVED_POLICY_VISITATIONS = budget / log2(k) / k * (k - 1)   (selfplay/src/main.rs:47-52)
    steps = k.bit_length() - 1
    return float(budget // steps // k * (k - 1))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return (float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1590.0))), "measured (bf16_tflops_sustained)",
                float(p.get("bf16_tflops", 0.0)) or None)
    return 1590.0, "fallback", None


def workload_config(wl: dict, name: str, n_gpus: int) -> dict:
    n = wl["n"]
    cfg = {
        "workload": name,
        "games_per_gpu": wl["games"], "games_total": wl["games"] * n_gpus,
        "sampled_actions": wl["k"], "search_budget": wl["budget"],
        "weights": "random init, torch seed 123, BN mean 0 / var 1, empty SimHash set",
        "l2": "inputs of every lock-step (node arenas of all games, queued positions and move lists) far larger than "
              "the 126 MB L2, no explicit flush; the network's chunk activation sets are L2-resident by design",
    }
    if wl["kind"] == "selfplay":
        cfg["description"] = (f"{n}x{n} Tak (half komi {HALF_KOMI}) self-play, {wl['games']} concurrent games per GPU, "
                              f"Gumbel sequential halving k={wl['k']}, {wl['budget']} sims/move, {20 if n == 5 else 16}x256 ResNet, "
                              f"model reload (weight generation) before every move")
        cfg["sharding"] = f"games sharded over {n_gpus} GPU(s) by contiguous global id, no data-path collective"
    else:
        cfg["description"] = (f"{n}x{n} Tak reanalyze: fresh-target search over a synthetic replay buffer of "
                              f"{wl['buffer']:,} positions (all plies of random playouts), batches of {wl['games']} fresh "
                              f"roots per GPU, k={wl['k']}, {wl['budget']} sims, 16x256 ResNet")
        cfg["sharding"] = (f"buffer positions sharded over {n_gpus} GPU(s) by contiguous index range, "
                           f"no data-path collective")
    return cfg


# ---------------------------------------------------------------------------------------- --dump-outputs

DUMP_GAMES = 1024  # at a move stride of 1024 this keeps a dump near 40 MB
DUMP_LIMIT = 64 << 20


def dump_games(G: int):
    """The games a dump keeps: all of them up to DUMP_GAMES, else the same seeded sample on every run."""
    import numpy as np

    if G <= DUMP_GAMES:
        return np.arange(G)
    return np.sort(np.random.default_rng(0).choice(G, size=DUMP_GAMES, replace=False))


def write_dump(directory: str, arrays: dict) -> None:
    """DIR/<name>.npy per array: floats as float32, integers as float32 when they have at most 16 bits (exact) and as
    float64 otherwise (exact up to 32 bits; 64-bit words are split into 32-bit halves before they get here)."""
    import numpy as np

    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        wide = a.dtype.kind in "iu" and a.dtype.itemsize > 2
        out[name] = np.ascontiguousarray(a, dtype=np.float64 if wide else np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def selfplay_outputs(m, rows) -> dict:
    """After tz_selfplay_move: the new positions (tz_get_positions) and the children of the new roots
    (tz_root_children), rows `rows`."""
    import numpy as np

    pos = m.positions()[rows]
    out = {"games": rows}
    # the 64-bit stack words as (low, high) 32-bit halves: exact in float64
    out["position_stack"] = np.ascontiguousarray(pos["stack"]).view(np.uint32)
    for f in ("height", "top", "to_move", "stones", "caps", "ply", "reversible_plies"):
        out[f"position_{f}"] = pos[f]
    tbl = m.root_children()
    tag, bits = tbl["eval_tag"][rows], tbl["eval_bits"][rows]
    out["root_n"] = tbl["n"][rows]
    for f in ("moves", "visits", "logit", "prob", "std_dev"):
        out[f"root_{f}"] = tbl[f][rows]
    out["root_eval_tag"] = tag
    # a VALUE evaluation holds an f32, a solved one (win / loss / draw) the ply count (exact in f32)
    out["root_eval"] = np.where(tag == 0, bits.view(np.float32), bits.astype(np.float32))
    return out


def reanalyze_outputs(m, rows) -> dict:
    """After tz_reanalyze_batch: the targets tz_reanalyze_read returns, rows `rows`."""
    t = m.reanalyze_read()
    return {"games": rows, **{f"target_{k}": v[rows] for k, v in t.items()}}


# ---------------------------------------------------------------------------------- restated reference (CPU)

def cpu_reference_setup(n: int):
    import torch

    from oracle import net_ref
    from oracle import oracle as O

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    net = net_ref.Net(n, seed=123)
    agent = net.as_oracle_agent()
    games = [O.new_opening(n, HALF_KOMI, (1000 + g) % 8, (1000 + g) // 8 % 2) for g in range(CPU_GAMES)]
    batched = O.Batched(games)
    betas = [0.0] * CPU_GAMES
    return batched, agent, betas, cores


def cpu_lockstep_rate(batched, agent, betas, min_seconds: float, min_locksteps: int):
    """Lock-step simulations of CPU_GAMES games (BatchedMCTS::simulate) until the time bound."""
    t0 = time.perf_counter()
    done = 0
    while done < min_locksteps or time.perf_counter() - t0 < min_seconds:
        batched.simulate(agent, betas)
        done += 1
    dt = time.perf_counter() - t0
    return CPU_GAMES * done / dt, done, dt


def run_reference(args, wl, emit):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = wl["n"]
    batched, agent, betas, cores = cpu_reference_setup(n)
    per_step = 2  # lock-step simulations per step: a bounded sample of one move's 1 + budget
    for _ in range(args.warmup):
        for _ in range(per_step):
            batched.simulate(agent, betas)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for _ in range(per_step):
            batched.simulate(agent, betas)
    dt = time.perf_counter() - t0
    value = CPU_GAMES * per_step * args.steps / dt
    sample = (f"{per_step} lock-step simulations of {CPU_GAMES} games per step (of the {1 + wl['budget']} one move "
              f"needs), from fresh roots, oracle C search + libtorch-CPU f32 forward")
    emit({
        "impl": "reference", "metric": wl["metric"], "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # what THIS arm times (not the GPU arm's workload): one reference process with its BATCH_SIZE of 128 games
        "config": {
            "workload": f"{args.workload} (restated reference, bounded sample)",
            "description": f"{n}x{n} Tak (half komi {HALF_KOMI}), ONE reference process: {CPU_GAMES} games in lock-step "
                           f"(BATCH_SIZE, selfplay/src/main.rs:37), {per_step} lock-step simulations per step from "
                           f"fresh roots, f32 16x256 ResNet on the host cores",
            "games_per_gpu": 0, "games_total": CPU_GAMES, "locksteps_per_step": per_step,
            "weights": "random init, torch seed 123, BN mean 0 / var 1, empty SimHash set",
            "same_config_as_gpu_arm": False,
        },
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "restated CPU baseline (oracle port), not the reference binary: no Rust toolchain in the image",
    })


# ---------------------------------------------------------------------------------------------- our arm

class Run:
    """Process-wide setup shared by the workloads: rank / device, process group, library, handle, communicator."""

    def __init__(self, args, wl):
        import torch

        from takzero_b200 import build as tz_build
        from takzero_b200 import capi, network, weights
        from takzero_b200 import distributed as tzd

        self.torch, self.capi, self.network, self.weights, self.tzd = torch, capi, network, weights, tzd
        self.args, self.wl = args, wl
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}: launch with torch.distributed.run")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (takzero_b200 has no CPU fallback)")
        torch.cuda.set_device(self.local_rank)
        self.cuda_dev = torch.device("cuda", self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=self.cuda_dev)
            self.dist = dist
        tz_build.build()
        n, G = wl["n"], wl["games"]
        game_base, _ = tzd.shard(self.rank, self.world, G)
        self.m = capi.BatchedMCTS(n, HALF_KOMI, G, device=self.local_rank, game_base=game_base)
        # the library's own NCCL communicator: weight generations and counter sums go through it
        tzd.init_comm(self.m, self.rank, self.world, self.cuda_dev if self.world > 1 else None)
        self.net_dtype = network.DTYPE_BF16 if os.environ.get("TZ_BENCH_DTYPE", "f16") == "bf16" else network.DTYPE_F16
        # the model of every generation: rank 0 owns the tensors (the others pass none)
        self.tensors = None
        if self.rank == 0:  # in pinned memory: the library then uploads them from where they are (no staging copy)
            self.tensors = {}
            for name, t in weights.random_init(n, seed=123).items():
                buf = capi.pinned_array(t.shape, "float32")
                buf[...] = t
                self.tensors[name] = buf
        self.raw_weight_bytes = sum(4 * v.size for v in self.tensors.values()) if self.tensors else 0
        t_w = time.perf_counter()
        self.generation()
        self.m.sync()
        self.first_generation_s = time.perf_counter() - t_w
        self.m.set_agent(capi.AGENT_NETWORK)
        self.peak, self.peak_kind, self.peak_burst = measured_peaks()
        self.flops_pos = weights.flops_per_position(n)

    def generation(self):
        """`Net::load` before a move (selfplay/src/main.rs:107) on all ranks: one tz_broadcast_weights."""
        self.network.broadcast_weights(self.m, self.tensors, root=0, dtype=self.net_dtype)

    def barrier(self):
        self.m.sync()
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, ms_list, counters):
        """max over ranks of device times, sums of counters (the library's ncclAllReduce)."""
        if self.dist is not None:
            ms_list = self.tzd.max_over_ranks(ms_list, self.cuda_dev)
            counters = self.network.allreduce_sum(self.m, [int(c) for c in counters])
        return ms_list, counters

    def roofline(self, prof):
        capi = self.capi
        cat = dict(zip(capi.PROFILE_CATEGORIES, range(8)))
        conv_ms = prof.ms[cat["conv_input"]] + prof.ms[cat["conv_tower"]] + prof.ms[cat["conv_policy"]]
        conv_launches = (prof.launches[cat["conv_input"]] + prof.launches[cat["conv_tower"]] +
                         prof.launches[cat["conv_policy"]])
        achieved = (prof.positions * self.flops_pos / (conv_ms / 1000.0) / 1e12) if conv_ms > 0 else 0.0
        traffic = None
        ncu_path = os.path.join(ROOT, "profiles", "conv_traffic.json")
        if os.path.exists(ncu_path) and self.args.workload != "4x4_1024":
            with open(ncu_path) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        dt = "fp16" if self.net_dtype == self.network.DTYPE_F16 else "bf16"
        return {
            "kernel": f"conv::k_conv3x3_pair ({dt} implicit GEMM, tcgen05 cta_group::2 / TMEM; one fused launch = the "
                      f"whole network pass: plane encoding, 34 convolutions, head features, legal-logit gather)",
            "bound": "tensor", "achieved": achieved,
            "peak": self.peak, "peak_kind": self.peak_kind, "unit": "TFLOP/s",
            "frac": achieved / self.peak if self.peak else None,
            # the kernel runs inside a long step, so the sustained cuBLAS rate is the denominator; against cuBLAS's
            # burst rate (a GEMM timed alone, before the power cap bites) the same number is:
            "peak_burst": self.peak_burst, "frac_of_burst": achieved / self.peak_burst if self.peak_burst else None,
            "traffic": traffic,
            "sampled": {"locksteps": int(prof.locksteps), "positions": int(prof.positions),
                        "conv_launches": int(conv_launches), "conv_ms": conv_ms,
                        "flop_per_position": self.flops_pos},
            "kernel_ms_sampled": {name: prof.ms[i] for name, i in cat.items() if prof.launches[i]},
        }

    def cpu_baseline(self):
        if self.world != 1 or self.args.no_cpu_baseline:
            return None
        batched, agent, cbetas, cores = cpu_reference_setup(self.wl["n"])
        batched.simulate(agent, cbetas)  # warm-up (root expansion, thread pool)
        rate, n_lock, dt = cpu_lockstep_rate(batched, agent, cbetas, 15.0, 4)
        return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{n_lock} lock-step simulations of {CPU_GAMES} games in {dt:.1f} s: oracle C search + "
                          f"libtorch-CPU f32 forward (torch threads = {cores}); restated reference, not the Rust binary"}

    def close(self):
        self.m.close()
        if self.dist is not None:
            self.dist.destroy_process_group()


def timed_selfplay(run: Run, params, steps: int, reload_every: int, profile: bool):
    """`steps` resident self-play moves with a weight generation before every `reload_every`-th one (0 = never)."""
    m = run.m
    run.barrier()
    c0, l0 = m.counters(), m.launch_count()
    if profile:
        m.profile_begin(8)
    gens = 0
    m.timer_start()
    for i in range(steps):
        if reload_every and i % reload_every == 0:
            run.generation()
            gens += 1
        m.selfplay_move(params)
    ms = m.timer_stop()
    gen_ms = run.network.weight_generation(m)[1] if gens else None
    run.barrier()
    prof = m.profile_end() if profile else None
    status = m.status()
    if status:
        raise SystemExit(f"device search error bits 0x{status:x} during the timed region")
    c1 = m.counters()
    return {"ms": ms, "sims": c1.simulations - c0.simulations, "evals": c1.evaluations - c0.evaluations,
            "known": c1.known - c0.known, "launches": m.launch_count() - l0, "generations": gens,
            "generation_ms": gen_ms, "prof": prof}


def run_selfplay(args, wl, emit):
    import numpy as np

    run = Run(args, wl)
    m, capi = run.m, run.capi
    G, k, budget, M = wl["games"], wl["k"], wl["budget"], run.m.move_stride
    vis = target_visitations(k, budget)
    params = capi.SelfplayParams(k, budget, 0.0, WEIGHTED_RANDOM_PLIES, SAMPLE_THRESHOLD, ALLOWED_DROP, vis,
                                 TARGET_BETA, 20261018)

    # ---- resident path: warm-up, then EXACTLY --steps timed moves, a weight generation before every move ----------
    def fresh_games():
        """Every timed loop searches the same plies: games from their openings + the warm-up moves."""
        m.new_openings(seed=1000)
        for _ in range(args.warmup):
            run.generation()
            m.selfplay_move(params)

    fresh_games()
    clocks = ClockSampler(run.local_rank)
    clocks.start()
    every = timed_selfplay(run, params, args.steps, 1, profile=True)
    clock_info = clocks.stop()
    if args.dump_outputs and run.rank == 0:
        write_dump(args.dump_outputs, selfplay_outputs(m, dump_games(G)))
    # the same with ONE generation in the region (the amortised cadence: a new model every >= --steps moves) and none
    fresh_games()
    sparse = timed_selfplay(run, params, args.steps, args.steps, profile=False)
    fresh_games()
    never = timed_selfplay(run, params, args.steps, 0, profile=False)
    positions = G * args.steps

    def rate(r):
        (ms,), (sims,) = run.reduce([r["ms"]], [r["sims"]])
        return sims / (ms / 1000.0), ms

    value, ms = rate(every)
    sparse_value, _ = rate(sparse)
    never_value, _ = rate(never)
    _, (sims, evals, known, positions, launches) = run.reduce(
        [0.0], [every["sims"], every["evals"], every["known"], positions, every["launches"]])
    (gen_ms,), _ = run.reduce([every["generation_ms"] or 0.0], [0])
    roofline = run.roofline(every["prof"])

    # ---- end to end through the host-buffer C ABI -------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        rng = np.random.default_rng(7 + run.rank)
        pool = 2
        gumbel_pool = capi.pinned_array((pool, G, M), np.float32)
        gumbel_pool[:] = rng.gumbel(size=(pool, G, M)).astype(np.float32)
        betas = capi.pinned_array((G,), np.float32)
        betas[:] = 0.0
        randoms = capi.pinned_array((G,), np.uint64)
        sym = capi.pinned_array((G,), np.int32)
        adj = capi.pinned_array((G,), np.int32)
        m.new_openings(seed=1000)  # the same plies as the resident loops
        plies = m.positions()["ply"].astype(np.int64)
        target_out = (capi.pinned_array((G, M), np.float32), capi.pinned_array((G,), np.float32),
                      capi.pinned_array((G,), np.int32))

        def host_move(i):
            nonlocal plies
            run.generation()  # Net::load: rank 0's f32 tensors go host -> device every move
            moves = m.gumbel_sequential_halving(betas, k, budget, gumbel_pool[i % pool])
            pol, ube, cnt = m.targets(vis, TARGET_BETA, out=target_out)
            randoms[:] = rng.integers(0, 1 << 62, size=G, dtype=np.uint64)
            sel = m.select_actions_in_selfplay(WEIGHTED_RANDOM_PLIES, SAMPLE_THRESHOLD, ALLOWED_DROP, randoms)
            play = np.where(plies < WEIGHTED_RANDOM_PLIES, sel, moves).astype(np.uint16)
            m.step(play)
            sym[:] = rng.integers(0, 8, size=G)
            adj[:] = rng.integers(0, 2, size=G)
            term = m.restart_terminal_envs(sym, adj)
            plies = np.where(term != 0, 2, plies + 1)
            return float(pol[0, 0]) + float(ube[0])

        h2d = 4 * G + 4 * G * M + 8 * G + 2 * G + 8 * G + run.raw_weight_bytes
        d2h = 2 * G + 4 * G * M + 4 * G + 4 * G + 2 * G + 4 * G + 5 * 4
        e2e_warm = max(1, args.warmup)
        for i in range(e2e_warm):
            host_move(i)
        run.barrier()
        ce0 = m.counters()
        t0 = time.perf_counter()
        m.timer_start()
        for i in range(args.steps):
            host_move(e2e_warm + i)
        ems = m.timer_stop()
        run.barrier()
        wall_ms = 1000.0 * (time.perf_counter() - t0)
        ce1 = m.counters()
        (ems, wall_ms), (esims,) = run.reduce([ems, wall_ms], [ce1.simulations - ce0.simulations])
        e2e = {"value": esims / (ems / 1000.0), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": ems / args.steps, "wall_ms_per_step": wall_ms / args.steps,
               "api": "tz_broadcast_weights + tz_gumbel_sequential_halving + tz_targets + tz_select_selfplay + tz_step + "
                      "tz_restart_terminal with pinned host buffers",
               "noise": "Gumbel noise injected from pinned host memory (the `value` leg draws it on the device)",
               "h2d_note": "rank 0's bytes: per-move noise / randoms / openings plus the model's f32 tensors of the "
                           "weight generation; the other ranks receive the 16-bit weight set over NCCL instead"}

    cpu = run.cpu_baseline()
    if run.rank == 0:
        cfg = workload_config(wl, args.workload, run.world)
        cfg["arena_slots_per_game"] = m.arena_slots
        cfg["first_generation_s"] = run.first_generation_s
        out = {
            "metric": wl["metric"], "value": value, "unit": UNIT, "n_gpus": run.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16" if run.net_dtype == run.network.DTYPE_F16 else "bf16",
            "data": "synthetic", "config": cfg,
            "positions_per_s": positions / (ms / 1000.0), "nn_evals_per_s": evals / (ms / 1000.0),
            "known_fraction": known / sims if sims else 0.0,
            "pipeline_tensor_frac": (evals / (ms / 1000.0)) * run.flops_pos / 1e12 / (run.peak * run.world),
            "gpu_launches": int(launches),
            # the model reload of selfplay/src/main.rs:107 as weight generations inside the timed region: `value` has
            # one before EVERY move; the same loop with one generation per --steps moves and with none for comparison
            "weight_generations": {
                "every_move": {"value": value, "generations": every["generations"]},
                "one_per_region": {"value": sparse_value, "generations": sparse["generations"]},
                "none": {"value": never_value, "generations": 0},
                # duration of the last generation on the side stream (upload + fold + broadcast; for N > 1 it includes
                # waiting for a gap between the search's network launches on every rank, because the NCCL kernel needs
                # SMs the persistent network kernel holds) and what a generation per move costs the timed loop
                "generation_ms_max_over_ranks": gen_ms,
                "cost_ms_per_move": (every["ms"] - never["ms"]) / args.steps,
                "what": "tz_broadcast_weights: f32 tensors H2D on rank 0, BatchNorm fold + arrangement on the GPU, "
                        "ncclBroadcast of the 16-bit set, swap between moves; on a side stream beside the search",
            },
            "clocks": clock_info, "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu,
        }
        emit(out)
    run.close()


def make_replay_buffer(run: Run, lo: int, hi: int):
    """This rank's index range [lo, hi) of the synthetic replay buffer: positions of random-playout games (uniform random
    legal moves from `new_opening`, every ply kept, like `Replay::states`, target.rs:205-212), generated on the device."""
    import numpy as np

    m = run.m
    want = hi - lo
    m.new_openings(seed=2000 + lo)
    chunks, have, it = [], 0, 0
    while have < want:
        pos = m.positions()
        live = m.result(pos) == 0
        chunks.append(pos[live])
        have += int(live.sum())
        m.random_steps(1, seed=2000 + it)
        done = (m.result(m.positions()) != 0).astype(np.uint8)
        if done.any():  # finished games start over from a new opening
            m.new_openings(seed=3000 + it, mask=done)
        it += 1
    buf = np.concatenate(chunks)[:want]
    buf["pad1"] = 0
    return buf


def run_reanalyze(args, wl, emit):
    import numpy as np

    run = Run(args, wl)
    m, capi = run.m, run.capi
    G, k, budget, M = wl["games"], wl["k"], wl["budget"], run.m.move_stride
    lo, hi = run.tzd.shard_range(wl["buffer"], run.rank, run.world)
    t0 = time.perf_counter()
    buffer = make_replay_buffer(run, lo, hi)
    m.stage_positions(buffer)
    buffer_s = time.perf_counter() - t0
    rng = np.random.default_rng(1 + run.rank)
    params = capi.ReanalyzeParams(k, budget, TARGET_BETA, 20261018)

    def sample():
        return rng.choice(len(buffer), size=G, replace=False).astype(np.uint32)

    # ---- resident: the staged buffer stays on the device, a batch picks its fresh roots by index ---------------------
    for _ in range(args.warmup):
        m.reanalyze_batch(sample(), params)
    run.barrier()
    c0, l0 = m.counters(), m.launch_count()
    clocks = ClockSampler(run.local_rank)
    clocks.start()
    m.profile_begin(8)
    m.timer_start()
    for _ in range(args.steps):
        m.reanalyze_batch(sample(), params)
    ms = m.timer_stop()
    run.barrier()
    prof = m.profile_end()
    clock_info = clocks.stop()
    if m.status():
        raise SystemExit(f"device search error bits 0x{m.status():x} during the timed region")
    c1 = m.counters()
    if args.dump_outputs and run.rank == 0:
        write_dump(args.dump_outputs, reanalyze_outputs(m, dump_games(G)))
    (ms,), (sims, evals, known, targets, launches) = run.reduce(
        [ms], [c1.simulations - c0.simulations, c1.evaluations - c0.evaluations, c1.known - c0.known, G * args.steps,
               m.launch_count() - l0])
    value = sims / (ms / 1000.0)
    roofline = run.roofline(prof)

    # ---- end to end: positions from host memory every batch, targets read back (what reanalyze's main loop does) -----
    e2e = None
    if not args.no_e2e:
        out = {"policy": capi.pinned_array((G, M), np.float32), "moves": capi.pinned_array((G, M), np.uint16),
               "ube": capi.pinned_array((G,), np.float32), "value": capi.pinned_array((G,), np.float32),
               "n": capi.pinned_array((G,), np.int32)}
        batch_states = capi.pinned_array((G,), capi.STATE_DTYPE)

        def host_batch():
            batch_states[:] = buffer[sample()]
            m.set_positions(batch_states)       # *node = Node::default(); *env = replay_env
            m.reanalyze_batch(None, params)
            t = m.reanalyze_read(out)
            return float(t["policy"][0, 0]) + float(t["ube"][0]) + float(t["value"][0])

        for _ in range(max(1, min(args.warmup, 2))):
            host_batch()
        run.barrier()
        ce0 = m.counters()
        w0 = time.perf_counter()
        m.timer_start()
        for _ in range(args.steps):
            host_batch()
        ems = m.timer_stop()
        run.barrier()
        wall_ms = 1000.0 * (time.perf_counter() - w0)
        ce1 = m.counters()
        (ems, wall_ms), (esims,) = run.reduce([ems, wall_ms], [ce1.simulations - ce0.simulations])
        e2e = {"value": esims / (ems / 1000.0), "unit": UNIT, "h2d_bytes_per_step": 384 * G,
               "d2h_bytes_per_step": 4 * G * M + 2 * G * M + 12 * G + 4,
               "ms_per_step": ems / args.steps, "wall_ms_per_step": wall_ms / args.steps,
               "targets_per_s": G * args.steps * run.world / (ems / 1000.0),
               "api": "tz_set_positions + tz_reanalyze_batch + tz_reanalyze_read with pinned host buffers"}

    cpu = run.cpu_baseline()
    if run.rank == 0:
        cfg = workload_config(wl, args.workload, run.world)
        cfg["arena_slots_per_game"] = m.arena_slots
        cfg["buffer_positions_total"] = wl["buffer"]
        cfg["buffer_positions_this_rank"] = int(len(buffer))
        cfg["buffer_generation_s"] = buffer_s
        cfg["positions_reanalyzed"] = int(targets)
        cfg["note"] = ("a step is one batch per GPU; --steps 16 at --gpus 8 reanalyzes 1,048,576 targets = one pass "
                       "over the buffer")
        emit({
            "metric": wl["metric"], "value": value, "unit": UNIT, "n_gpus": run.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16" if run.net_dtype == run.network.DTYPE_F16 else "bf16",
            "data": "synthetic", "config": cfg,
            "targets_per_s": targets / (ms / 1000.0), "positions_per_s": targets / (ms / 1000.0),
            "nn_evals_per_s": evals / (ms / 1000.0), "known_fraction": known / sims if sims else 0.0,
            "pipeline_tensor_frac": (evals / (ms / 1000.0)) * run.flops_pos / 1e12 / (run.peak * run.world),
            "gpu_launches": int(launches), "clocks": clock_info, "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu,
        })
    run.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="6x6_selfplay", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA library's outputs: it needs --impl ours")
    wl = WORKLOADS[args.workload]
    # stdout carries exactly ONE line, the JSON result: anything a library prints on the way (NCCL's version
    # banner, torchrun notices) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(json_fd, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    if args.impl == "reference":
        run_reference(args, wl, emit)
    elif wl["kind"] == "selfplay":
        run_selfplay(args, wl, emit)
    else:
        run_reanalyze(args, wl, emit)


if __name__ == "__main__":
    main()
