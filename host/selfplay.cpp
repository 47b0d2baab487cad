// selfplay.cpp -- the reference's `selfplay` binary (selfplay/src/main.rs:63-203) as a C++ host over
// libtakzero_b200.so: search every game with Gumbel sequential halving, sample early plies by visits,
// record improved-policy / UBE targets, step, restart finished games, complete their value targets by
// walking the result back (main.rs:263-329) and append `targets-selfplay.txt` / `replays.txt` in the
// reference's text formats (target.rs:56-73,215-232) so `learn` can consume them unchanged.
//
// Differences from the reference, all at the process boundary: constants are flags instead of
// compile-time consts (main.rs:36-52); the model is `--weights` or <directory>/model_latest.ot (the tch archive
// `learn` writes, read without libtorch; a TZW1 file `model_latest.tzw` is the second choice), re-read before a
// move whenever the file changed (the reference reloads unconditionally every move, main.rs:107); the
// `buffer_lengths.txt` throttle with its checksum (main.rs:93-104,371-387) is honoured when that file exists;
// the loop stops after --moves iterations.  Several GPUs: one process per GPU with `--device d --game-base d*games`,
// all appending to the same files like the reference's independent processes (README.md:128-130).
//
// --resident runs the same loop with tz_selfplay_move and the library's on-device training-data records
// (tz_selfplay_record / tz_selfplay_read): one asynchronous call per move instead of five blocking ones and no
// full-stride target table on the host; the text of one move is formatted while the device searches the next.
// Both modes write byte-identical files.  --record-bytes sets the record region per game (0: the library default).
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "../include/takzero_b200.hpp"

using namespace takzero;

struct IncompleteTarget {  // main.rs:230-234
    tz_state_t env;
    std::vector<std::pair<Move, float>> policy;
    float root_ube_metric;
};

struct Args {
    std::string directory = ".";
    std::string weights;  // empty: synthetic agent (deterministic hash, for tests)
    int board = 6, half_komi = 4, games = 128, device = 0, moves = 1;
    int game_base = 0;  // global id of game 0: one process per GPU, each with its own range (distinct RNG streams)
    int sampled_actions = 64, weighted_random_plies = 10;
    unsigned budget = 768;
    unsigned long long seed = 1;
    float beta = 0.25f;
    bool exploration = false;
    bool resident = false;
    unsigned arena_slots = 0;
    unsigned long long record_bytes = 0;
};

static Args parse(int argc, char** argv) {
    Args a;
    for (int i = 1; i < argc; i++) {
        const std::string k = argv[i];
        auto val = [&]() -> const char* {
            if (i + 1 >= argc) {
                std::fprintf(stderr, "missing value for %s\n", k.c_str());
                std::exit(2);
            }
            return argv[++i];
        };
        if (k == "--directory") a.directory = val();
        else if (k == "--weights") a.weights = val();
        else if (k == "--board") a.board = std::atoi(val());
        else if (k == "--half-komi") a.half_komi = std::atoi(val());
        else if (k == "--games") a.games = std::atoi(val());
        else if (k == "--device") a.device = std::atoi(val());
        else if (k == "--game-base") a.game_base = std::atoi(val());
        else if (k == "--moves") a.moves = std::atoi(val());
        else if (k == "--sampled-actions") a.sampled_actions = std::atoi(val());
        else if (k == "--budget") a.budget = (unsigned)std::atoi(val());
        else if (k == "--weighted-random-plies") a.weighted_random_plies = std::atoi(val());
        else if (k == "--seed") a.seed = std::strtoull(val(), nullptr, 10);
        else if (k == "--arena-slots") a.arena_slots = (unsigned)std::atoi(val());
        else if (k == "--exploration") a.exploration = true;
        else if (k == "--resident") a.resident = true;
        else if (k == "--record-bytes") a.record_bytes = std::strtoull(val(), nullptr, 10);
        else {
            std::fprintf(stderr, "unknown flag %s\n", k.c_str());
            std::exit(2);
        }
    }
    return a;
}

static const size_t MAX_SELFPLAY_BUFFER_LEN = 32000;  // main.rs:43

static void append(const std::string& path, const std::string& contents) {
    if (!append_file(path, contents))
        std::fprintf(stderr, "Could not save to %s, so here it is instead:\n%s", path.c_str(), contents.c_str());
}

int main(int argc, char** argv) {
    Args args = parse(argc, argv);
    try {
        BatchedMCTS mcts(args.board, args.half_komi, args.games, args.device, args.game_base, args.arena_slots);
        for (const char* name : {"/model_latest.ot", "/model_latest.tzw"})
            if (args.weights.empty() && mtime_ns(args.directory + name) >= 0) args.weights = args.directory + name;
        long long model_stamp = -1;
        auto reload_model = [&]() {  // Net::load before every move (main.rs:107), skipped while unchanged
            if (args.weights.empty()) return;
            const long long stamp = mtime_ns(args.weights);
            if (stamp == model_stamp) return;
            try {
                mcts.load_model(args.weights);
                mcts.set_agent(TZ_AGENT_NETWORK);
                model_stamp = stamp;
            } catch (const std::exception& e) {
                if (model_stamp < 0) throw;  // no model at all yet
                std::fprintf(stderr, "Cannot load model: %s, keeping the previous one.\n", e.what());
            }
        };
        reload_model();
        mcts.new_openings(args.seed);  // BatchedMCTS::new -> Env::new_opening
        const int G = args.games, n = args.board, stride = mcts.move_stride();
        // `exploration` feature: the first half of the batch searches with BETA (main.rs:81-87)
        std::vector<float> betas(G, 0.0f);
        if (args.exploration)
            for (int g = 0; g < G / 2; g++) betas[g] = args.beta;
        // IMPROVED_POLICY_VISITATIONS (main.rs:47-52)
        unsigned log_sampled = 0;
        while ((2u << log_sampled) <= (unsigned)args.sampled_actions) log_sampled++;
        const unsigned visitations = args.budget / log_sampled / (unsigned)args.sampled_actions * ((1u << log_sampled) - 1);

        // wait while the trainer's exploitation buffer is full (main.rs:93-104)
        auto throttle = [&]() {
            for (;;) {
                const BufferLengths lengths = read_buffer_lengths(args.directory);
                if (lengths.status == -1 || (lengths.status == 0 && lengths.selfplay <= MAX_SELFPLAY_BUFFER_LEN)) break;
                if (lengths.status == -2) std::fprintf(stderr, "Could not read buffer lengths: wrong checksum or missing component\n");
                std::this_thread::sleep_for(std::chrono::seconds(1));
            }
        };

        if (args.resident) {
            mcts.selfplay_record(true, (size_t)args.record_bytes);
            tz_selfplay_t sp{};
            sp.sampled_actions = args.sampled_actions;
            sp.search_budget = args.budget;
            sp.beta = args.exploration ? args.beta : 0.0f;
            sp.weighted_random_plies = args.weighted_random_plies;
            sp.sample_threshold = 32;
            sp.allowed_eval_drop = 0.5f;
            sp.target_visitations = (float)visitations;
            sp.target_beta = args.beta;
            sp.seed = args.seed;
            bool warned_full = false;
            // restart_envs_and_complete_targets' file output (main.rs:263-329) of one move's data
            auto write = [&](const BatchedMCTS::SelfplayData& data) {
                std::string targets_txt, replays_txt, exploration_txt;
                for (const BatchedMCTS::FinishedGame& f : data.games) {
                    if (args.exploration && f.exploration) {
                        Replay head = f.replay;
                        if ((int)head.actions.size() > args.weighted_random_plies) head.actions.resize(args.weighted_random_plies);
                        exploration_txt += head.to_string(n, head.actions.size() == f.replay.actions.size() ? f.result : 0);
                    }
                    replays_txt += f.replay.to_string(n, f.result);
                }
                for (const Target& t : data.targets) targets_txt += t.to_string(n);
                if (!targets_txt.empty()) append(args.directory + "/targets-selfplay.txt", targets_txt);
                if (!replays_txt.empty()) append(args.directory + "/replays.txt", replays_txt);
                if (!exploration_txt.empty()) append(args.directory + "/replays-exploration.txt", exploration_txt);
            };
            BatchedMCTS::SelfplayData prev;
            bool have_prev = false;
            for (int step = 0; step < args.moves; step++) {
                throttle();
                reload_model();
                mcts.selfplay_move(sp);
                if (have_prev) write(prev);  // formatted while the device searches this move
                prev = mcts.selfplay_read();
                have_prev = true;
                uint32_t bits = 0;
                check(tz_status(mcts.handle(), &bits));
                if (bits & TZ_STATUS_TARGETS_FULL) {
                    if (!warned_full)
                        std::fprintf(stderr, "selfplay: training data dropped (record region or queue full, high-water "
                                             "mark %zu bytes per game); raise --record-bytes\n", prev.high_water_bytes);
                    warned_full = true;
                    check(tz_clear_status(mcts.handle()));
                }
            }
            if (have_prev) write(prev);
            const tz_counters_t c = mcts.counters();
            std::printf("selfplay: %d moves of %d games, %llu simulations, %llu evaluations\n", args.moves, G,
                        (unsigned long long)c.simulations, (unsigned long long)c.evaluations);
            return 0;
        }

        std::vector<std::vector<IncompleteTarget>> policy_targets(G);
        std::vector<tz_state_t> cur = mcts.envs();
        for (int step = 0; step < args.moves; step++) {
            throttle();
            reload_model();
            std::vector<Move> selected =
                mcts.gumbel_sequential_halving(betas, args.sampled_actions, args.budget, args.seed);
            const std::vector<Move> sampled = mcts.select_actions_in_selfplay(args.weighted_random_plies, args.seed);
            for (int g = 0; g < G; g++)
                if ((int)cur[g].ply < args.weighted_random_plies) selected[g] = sampled[g];  // main.rs:143-152
            // take_a_step (main.rs:238-258)
            const BatchedMCTS::RootTargets rt = mcts.targets((float)visitations, args.beta);
            for (int g = 0; g < G; g++) {
                IncompleteTarget t;
                t.env = cur[g];
                for (int i = 0; i < rt.n[g]; i++)
                    t.policy.emplace_back(rt.moves[(size_t)g * stride + i], rt.policy[(size_t)g * stride + i]);
                t.root_ube_metric = rt.ube[g];
                policy_targets[g].push_back(std::move(t));
            }
            mcts.step(selected);
            const std::vector<tz_state_t> after = mcts.envs();
            // restart_envs_and_complete_targets (main.rs:263-329)
            const std::vector<int> terminal = mcts.restart_terminal_envs(args.seed);
            std::string targets_txt, replays_txt, exploration_txt;
            std::vector<int> finished;
            std::vector<tz_state_t> finals;
            for (int g = 0; g < G; g++)
                if (terminal[g]) {
                    finished.push_back(g);
                    finals.push_back(after[g]);
                }
            std::vector<int> results(finished.size());
            if (!finished.empty()) check(tz_game_result(mcts.handle(), finals.data(), (int)finals.size(), results.data()));
            for (size_t k = 0; k < finished.size(); k++) {
                const int g = finished[k];
                const Replay replay = mcts.finished_replay(g);
                if (args.exploration && betas[g] > 0.0f) {
                    Replay head = replay;
                    if ((int)head.actions.size() > args.weighted_random_plies) head.actions.resize(args.weighted_random_plies);
                    // the truncated replay is re-evaluated by Display, which prints a result only if the
                    // truncated game is over; early plies never are
                    exploration_txt += head.to_string(n, (int)head.actions.size() == (int)replay.actions.size() ? results[k] : 0);
                }
                replays_txt += replay.to_string(n, results[k]);
                Eval value = Eval::from_terminal(terminal[g]);
                for (auto it = policy_targets[g].rbegin(); it != policy_targets[g].rend(); ++it) {
                    value = value.negate();
                    if (betas[g] == 0.0f || (int)it->env.ply > args.weighted_random_plies) {
                        Target t;
                        t.env = it->env;
                        t.policy = std::move(it->policy);
                        t.value = value.to_f32();
                        t.ube = it->root_ube_metric;
                        targets_txt += t.to_string(n);
                    }
                }
                policy_targets[g].clear();
            }
            if (!targets_txt.empty()) append(args.directory + "/targets-selfplay.txt", targets_txt);
            if (!replays_txt.empty()) append(args.directory + "/replays.txt", replays_txt);
            if (!exploration_txt.empty()) append(args.directory + "/replays-exploration.txt", exploration_txt);
            cur = mcts.envs();
        }
        const tz_counters_t c = mcts.counters();
        std::printf("selfplay: %d moves of %d games, %llu simulations, %llu evaluations\n", args.moves, G,
                    (unsigned long long)c.simulations, (unsigned long long)c.evaluations);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "selfplay: %s\n", e.what());
        return 1;
    }
    return 0;
}
