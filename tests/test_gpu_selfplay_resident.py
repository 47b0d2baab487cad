"""GPU: resident self-play keeps its training data (tz_selfplay_record / tz_selfplay_read).

Every target and replay that tz_selfplay_move emits must equal, bit for bit, what the host-buffer loop of
host/selfplay.cpp (selfplay/src/main.rs:138-153,238-329) produces from a second handle with the same seed: search,
sample, targets, step, restart, finished replays, and the value walk-back done here in Python through the oracle's
Eval.  Both handles draw from the same RNG counters, so their searches are identical."""
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from takzero_b200 import build as tz_build
from takzero_b200 import capi

pytestmark = pytest.mark.gpu


def bits(x) -> int:
    return int(np.float32(x).view(np.uint32))


def params(k, budget, seed, plies=10, beta=0.0, target_beta=0.25):
    steps = k.bit_length() - 1
    vis = float(budget // steps // k * ((1 << steps) - 1))  # IMPROVED_POLICY_VISITATIONS (main.rs:47-52)
    return capi.SelfplayParams(k, budget, beta, plies, 32, 0.5, vis, target_beta, seed)


def make(n, G, seed, game_base=0, agent=None, random_steps=0):
    m = capi.BatchedMCTS(n, 4, G, game_base=game_base, arena_slots=1 << 15)
    m.new_openings(seed=seed)
    if random_steps:
        m.random_steps(random_steps, seed=seed)
        m.restart_terminal_envs(seed=seed)  # no game starts over (late positions: reserves run low)
    if agent is not None:
        agent(m)
    return m


def resident_records(d):
    """(targets, replays) of one tz_selfplay_read as comparable tuples, in emission order."""
    targets, replays = [], []
    for i in range(d["n_targets"]):
        o, n = int(d["target_offset"][i]), int(d["target_n"][i])
        targets.append((int(d["target_game"][i]), d["target_env"][i].tobytes(), bits(d["target_value"][i]),
                        bits(d["target_ube"][i]), d["policy_moves"][o:o + n].tobytes(),
                        d["policy_probs"][o:o + n].view(np.uint32).tobytes()))
    for j in range(d["n_replays"]):
        o, L = int(d["replay_offset"][j]), int(d["replay_length"][j])
        replays.append((int(d["replay_game"][j]), d["replay_start"][j].tobytes(), d["replay_moves"][o:o + L].tobytes(),
                        int(d["replay_result"][j]), int(d["replay_exploration"][j])))
    return targets, replays


class HostLoop:
    """The host-buffer sequence of host/selfplay.cpp, one move per call, on its own handle."""

    def __init__(self, m, sp, exploration=False):
        self.m, self.sp = m, sp
        self.betas = np.zeros(m.G, dtype=np.float32)
        if exploration:
            self.betas[: m.G // 2] = sp.beta
        self.pending = [[] for _ in range(m.G)]
        self.base = m.game_base

    def move(self):
        m, sp = self.m, self.sp
        cur = m.positions()
        selected = m.gumbel_sequential_halving(self.betas, sp.sampled_actions, sp.search_budget, None, seed=sp.seed)
        sampled = m.select_actions_in_selfplay(sp.weighted_random_plies, 32, 0.5, None, seed=sp.seed)
        selected = np.where(cur["ply"] < sp.weighted_random_plies, sampled, selected).astype(np.uint16)
        pol, ube, cnt, mv = m.targets(sp.target_visitations, sp.target_beta, with_moves=True)
        for g in range(m.G):
            c = int(cnt[g])
            self.pending[g].append((cur[g].copy(), mv[g, :c].tobytes(), pol[g, :c].view(np.uint32).tobytes(),
                                    bits(ube[g])))
        m.step(selected)
        after = m.positions()
        term = m.restart_terminal_envs(seed=sp.seed)
        fin = [g for g in range(m.G) if term[g]]
        results = m.game_result(after[fin]) if fin else []
        targets, replays = [], []
        for j, g in enumerate(fin):
            start, actions = m.finished_replay(g)
            replays.append((self.base + g, start.tobytes(), actions.astype(np.uint16).tobytes(), int(results[j]),
                            int(self.betas[g] > 0)))
            value = O.make_eval(int(term[g]), 0)
            for env, moves, probs, u in reversed(self.pending[g]):
                value = O.lib().tk_eval_negate(value)
                if self.betas[g] == 0 or int(env["ply"]) > sp.weighted_random_plies:
                    targets.append((self.base + g, env.tobytes(), bits(O.lib().tk_eval_to_f32(value)), u, moves, probs))
            self.pending[g] = []
        return targets, replays

    def clear(self):
        self.pending = [[] for _ in range(self.m.G)]


def run_pair(n, G, k, budget, moves, seed, beta=0.0, agent=None, random_steps=0):
    a = make(n, G, seed, agent=agent, random_steps=random_steps)
    b = make(n, G, seed, agent=agent, random_steps=random_steps)
    a.selfplay_record(True)
    sp = params(k, budget, seed, beta=beta)
    host = HostLoop(b, sp, exploration=beta != 0.0)
    got_t, got_r, want_t, want_r = [], [], [], []
    for _ in range(moves):
        a.selfplay_move(sp)
        t, r = resident_records(a.selfplay_read())
        got_t += t
        got_r += r
        t, r = host.move()
        want_t += t
        want_r += r
    assert a.status() == 0 and b.status() == 0
    assert (a.positions().tobytes() == b.positions().tobytes())
    a.close()
    b.close()
    return got_t, got_r, want_t, want_r


def _network_agent(n, seed):
    def agent(m):
        from takzero_b200 import network, weights

        network.set_weights(m, weights.random_init(n, seed=seed, blocks=2))
        m.set_agent(capi.AGENT_NETWORK)
    return agent


@pytest.mark.parametrize("case", ["4x4", "3x3_long", "exploration", "6x6_network"])
def test_resident_records_equal_the_host_loop(case):
    if case == "4x4":
        got_t, got_r, want_t, want_r = run_pair(4, 32, 8, 48, 70, 5)
    elif case == "3x3_long":
        got_t, got_r, want_t, want_r = run_pair(3, 16, 4, 16, 120, 11)
    elif case == "exploration":
        got_t, got_r, want_t, want_r = run_pair(4, 32, 8, 48, 70, 7, beta=0.25)
        assert any(r[4] for r in got_r) and any(not r[4] for r in got_r)
    else:
        got_t, got_r, want_t, want_r = run_pair(6, 32, 8, 48, 80, 3, agent=_network_agent(6, 2), random_steps=52)
    assert len(got_r) >= 3, "the run must finish some games"
    assert len(got_r) == len(want_r) and got_r == want_r
    assert len(got_t) == len(want_t)
    for i, (g, w) in enumerate(zip(got_t, want_t)):
        assert g == w, f"target {i} (game {w[0]}) differs"


def test_recording_does_not_perturb_the_search():
    n, G, k, budget, moves, seed = 4, 32, 8, 48, 25, 9
    on, off, toggled = make(n, G, seed), make(n, G, seed), make(n, G, seed)
    on.selfplay_record(True)
    toggled.selfplay_record(True)
    toggled.selfplay_record(False)
    sp = params(k, budget, seed)
    for _ in range(moves):
        for m in (on, off, toggled):
            m.selfplay_move(sp)
    ref = off.root_children()
    for m in (on, toggled):
        assert m.positions().tobytes() == off.positions().tobytes()
        ch = m.root_children()
        for key in ref:
            assert np.array_equal(ch[key], ref[key]), key
        c, r = m.counters(), off.counters()
        assert (c.simulations, c.evaluations, c.known, c.expansions) == (r.simulations, r.evaluations, r.known,
                                                                           r.expansions)
    # launches of a move with recording off: 1 + 49 lock-steps x 3 + (2 + log2 k) + 5 (api.cu tz_selfplay_move)
    per_move = 1 + (budget + 1) * 3 + 2 + 3 + 5
    assert off.launch_count() == toggled.launch_count() == moves * per_move
    assert on.launch_count() == moves * (per_move + 4)
    for m in (on, off, toggled):
        m.close()


def test_sharded_handles_give_the_same_records_per_game():
    n, G, k, budget, moves, seed = 4, 32, 8, 48, 60, 13
    one = make(n, G, seed)
    halves = [make(n, G // 2, seed, game_base=base) for base in (0, G // 2)]
    sp = params(k, budget, seed)
    per_game = [{}, {}]
    for i, handles in enumerate(([one], halves)):
        for m in handles:
            m.selfplay_record(True)
        for _ in range(moves):
            for m in handles:
                m.selfplay_move(sp)
            for m in handles:
                t, r = resident_records(m.selfplay_read())
                for rec in t + r:
                    per_game[i].setdefault(rec[0], []).append(rec)
        for m in handles:
            m.close()
    assert len(per_game[0]) >= 5
    assert per_game[0] == per_game[1]


def test_full_record_region_keeps_the_prefix():
    n, G, k, budget, moves, seed = 4, 32, 8, 48, 70, 5
    full = make(n, G, seed)
    tiny = make(n, G, seed)
    full.selfplay_record(True)
    tiny.selfplay_record(True, bytes_per_game=4096)
    sp = params(k, budget, seed)
    got, want = [], []
    for _ in range(moves):
        full.selfplay_move(sp)
        tiny.selfplay_move(sp)
        ft, fr = resident_records(full.selfplay_read())
        d = tiny.selfplay_read()
        assert d["high_water_bytes"] <= 4096
        tt, tr = resident_records(d)
        assert tr == fr
        for g in sorted({r[0] for r in fr}):
            want.append([t for t in ft if t[0] == g])
            got.append([t for t in tt if t[0] == g])
    assert tiny.status() & capi.STATUS_TARGETS_FULL
    assert full.status() == 0
    assert tiny.positions().tobytes() == full.positions().tobytes()
    assert any(len(g) < len(w) for g, w in zip(got, want))
    for g, w in zip(got, want):
        assert g == w[len(w) - len(g):]  # records of the first plies = the tail (last ply first)
    full.close()
    tiny.close()


def test_small_read_capacity_consumes_nothing():
    n, G, k, budget, moves, seed = 4, 32, 8, 48, 40, 5
    a, b = make(n, G, seed), make(n, G, seed)
    a.selfplay_record(True)
    sp = params(k, budget, seed)
    host = HostLoop(b, sp)
    want_t, want_r = [], []
    for _ in range(moves):  # the queue accumulates
        a.selfplay_move(sp)
        t, r = host.move()
        want_t += t
        want_r += r
    assert want_r
    cap = {"n_targets": len(want_t) - 1, "n_policy": 1 << 20, "n_replays": 1 << 10, "n_moves": 1 << 16}
    with pytest.raises(capi.TakzeroError, match="capacity too small"):
        a.selfplay_read(cap)
    got_t, got_r = resident_records(a.selfplay_read())
    assert got_r == want_r and got_t == want_t
    empty = a.selfplay_read()
    assert empty["n_targets"] == 0 and empty["n_replays"] == 0
    a.close()
    b.close()


def test_host_step_between_resident_moves_clears_pending_records():
    n, G, k, budget, seed = 4, 32, 8, 48, 17
    a, b = make(n, G, seed), make(n, G, seed)
    a.selfplay_record(True)
    sp = params(k, budget, seed)
    host = HostLoop(b, sp)
    got_t, got_r, want_t, want_r = [], [], [], []

    def both_moves(count):
        for _ in range(count):
            a.selfplay_move(sp)
            t, r = resident_records(a.selfplay_read())
            got_t.extend(t)
            got_r.extend(r)
            t, r = host.move()
            want_t.extend(t)
            want_r.extend(r)

    both_moves(6)
    for m in (a, b):  # one host step and restart on both handles; pending records describe stale positions now
        m.simulate(None)  # restarted games have fresh roots without children
        m.step(m.select_best_actions())
        m.restart_terminal_envs(seed=seed)
    host.clear()
    both_moves(40)
    assert got_r and got_r == want_r and got_t == want_t
    a.close()
    b.close()


def _run_selfplay(exe, directory, flags, resident):
    out = subprocess.run([exe, "--directory", str(directory), *flags] + (["--resident"] if resident else []),
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr
    return out.stdout


FILES = ("targets-selfplay.txt", "replays.txt", "replays-exploration.txt")


def _read(d, name):
    p = d / name
    return p.read_bytes() if p.exists() else None


@pytest.mark.parametrize("exploration", [False, True])
def test_resident_binary_writes_identical_files(tmp_path, exploration):
    tz_build.build()
    exe = os.path.join(os.path.dirname(capi.LIB_PATH), "bin", "selfplay")
    n, hk, G, k, budget, moves, seed = 4, 4, 32, 8, 48, 70, 5
    flags = ["--board", str(n), "--half-komi", str(hk), "--games", str(G), "--sampled-actions", str(k), "--budget",
             str(budget), "--moves", str(moves), "--seed", str(seed), "--arena-slots", str(1 << 15)]
    if exploration:
        flags.append("--exploration")
    dirs = [tmp_path / "host", tmp_path / "resident"]
    outs = []
    for d, resident in zip(dirs, (False, True)):
        d.mkdir()
        outs.append(_run_selfplay(exe, d, flags, resident))
    assert outs[0] == outs[1]
    for name in FILES:
        assert _read(dirs[0], name) == _read(dirs[1], name), name
    assert _read(dirs[1], "replays.txt").count(b"\n") >= 5
    if exploration:
        assert _read(dirs[1], "replays-exploration.txt")
    else:
        from test_gpu_selfplay_host import python_selfplay  # third witness: Python + oracle formatting

        want_targets, want_replays = python_selfplay(n, hk, G, k, budget, moves, seed)
        assert _read(dirs[1], "targets-selfplay.txt").decode() == want_targets
        assert _read(dirs[1], "replays.txt").decode() == want_replays


def test_resident_binary_with_network_weights_and_buffer_file(tmp_path):
    from takzero_b200 import weights

    tz_build.build()
    exe = os.path.join(os.path.dirname(capi.LIB_PATH), "bin", "selfplay")
    w = weights.random_init(4, seed=1, blocks=2)
    flags = ["--board", "4", "--half-komi", "4", "--games", "64", "--sampled-actions", "8", "--budget", "48",
             "--moves", "40", "--seed", "3", "--arena-slots", str(1 << 15)]
    dirs = [tmp_path / "host", tmp_path / "resident"]
    outs = []
    for d, resident in zip(dirs, (False, True)):
        d.mkdir()
        weights.save_tzw(str(d / "model_latest.tzw"), w)
        (d / "buffer_lengths.txt").write_text("100,50,150")  # selfplay, reanalyze, checksum: below the limit
        outs.append(_run_selfplay(exe, d, flags, resident))
    assert outs[0] == outs[1] and f"{64 * 40 * 49} simulations" in outs[1]
    for name in FILES:
        assert _read(dirs[0], name) == _read(dirs[1], name), name
    assert _read(dirs[1], "targets-selfplay.txt")
