// analysis.cpp -- the reference's `analysis` REPL (analysis/src/main.rs) as a C++ host over libtakzero_b200.so: one
// search tree (game 0 of a handle) that the user steers from stdin.  A line that parses as a move is played
// (`env.play` + `Node::descend`: the explored sub-tree is kept); any other line runs `simulate_batch(agent, env,
// BETA = 0, BATCH_SIZE = 128)`; after either, the root is printed with `impl Display for Node` (node/debug.rs).
// `--example` plays a whole game against itself: simulate, `select_best_action`, descend (main.rs:33-42).
// `--positions FILE --batches K` analyses a list of positions instead (one TPS per line; blank lines are skipped): each
// position is the tree of one game of a single handle, all trees get K simulate_batch calls side by side
// (tz_trees_simulate_batch, one network batch for all of them), then, in file order, every position prints its TPS, its
// root as the REPL would and its principal variation.
// Differences at the process boundary: --model-path may be omitted (deterministic synthetic agent, for tests);
// board size and komi are flags; end of input ends the program.
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

#include "../include/takzero_b200.hpp"

using namespace takzero;

static const float BETA = 0.0f;

// one position per non-blank line; false (with the line number on stderr) at the first line that is not TPS
static bool read_positions(const std::string& path, int board, std::vector<tz_state_t>* out) {
    std::ifstream in(path);
    if (!in) {
        std::fprintf(stderr, "analysis: cannot read %s\n", path.c_str());
        return false;
    }
    std::string line;
    for (int no = 1; std::getline(in, line); no++) {
        const size_t a = line.find_first_not_of(" \t\r\n"), b = line.find_last_not_of(" \t\r\n");
        if (a == std::string::npos) continue;
        tz_state_t env;
        if (!parse_tps(line.substr(a, b - a + 1), board, &env)) {
            std::fprintf(stderr, "analysis: %s line %d is not valid TPS\n", path.c_str(), no);
            return false;
        }
        out->push_back(env);
    }
    if (out->empty()) {
        std::fprintf(stderr, "analysis: %s holds no position\n", path.c_str());
        return false;
    }
    return true;
}

static int analyse_positions(const std::vector<tz_state_t>& envs, int board, int half_komi, int device,
                             unsigned arena_slots, int batch_size, int batches, const std::string& model_path) {
    const int count = (int)envs.size();
    BatchedMCTS mcts(board, half_komi, count, device, 0, arena_slots, count * batch_size);
    if (!model_path.empty()) {
        mcts.load_model(model_path);
        mcts.set_agent(TZ_AGENT_NETWORK);
    }
    mcts.set_positions(envs);
    for (int k = 0; k < batches; k++) mcts.trees_simulate_batch(BETA, batch_size);
    const std::vector<std::vector<Move>> pv = mcts.trees_principal_variation();
    for (int g = 0; g < count; g++) {
        std::cout << "tps: " << tps(envs[g], board) << "\n" << node_display(mcts, g) << "pv:";
        for (Move m : pv[g]) std::cout << ' ' << move_to_string(m);
        std::cout << "\n";
    }
    return 0;
}

int main(int argc, char** argv) {
    int board = 6, half_komi = 4, device = 0, batch_size = 128;
    unsigned arena_slots = 1u << 22;
    std::string model_path, tps_text, positions_path;
    int batches = -1;
    bool example = false;
    for (int i = 1; i < argc; i++) {
        const std::string k = argv[i];
        if (k == "--example") {
            example = true;
            continue;
        }
        if (i + 1 >= argc) {
            std::fprintf(stderr, "missing value for %s\n", k.c_str());
            return 2;
        }
        const char* v = argv[++i];
        if (k == "--model-path") model_path = v;
        else if (k == "--tps") tps_text = v;
        else if (k == "--board") board = std::atoi(v);
        else if (k == "--half-komi") half_komi = std::atoi(v);
        else if (k == "--device") device = std::atoi(v);
        else if (k == "--batch-size") batch_size = std::atoi(v);
        else if (k == "--arena-slots") arena_slots = (unsigned)std::atoi(v);
        else if (k == "--positions") positions_path = v;
        else if (k == "--batches") batches = std::atoi(v);
        else {
            std::fprintf(stderr, "unknown flag %s\n", k.c_str());
            return 2;
        }
    }
    if (!positions_path.empty() || batches >= 0) {
        if (positions_path.empty() || batches < 1 || example || !tps_text.empty()) {
            std::fprintf(stderr, "analysis: --positions FILE needs --batches K >= 1 and neither --example nor --tps\n");
            return 2;
        }
        if (board < 3 || board > 6 || batch_size < 1) {
            std::fprintf(stderr, "analysis: --board must be 3..6 and --batch-size >= 1\n");
            return 2;
        }
        std::vector<tz_state_t> envs;
        if (!read_positions(positions_path, board, &envs)) return 2;
        try {
            return analyse_positions(envs, board, half_komi, device, arena_slots, batch_size, batches, model_path);
        } catch (const std::exception& e) {
            std::fprintf(stderr, "analysis: %s\n", e.what());
            return 1;
        }
    }
    try {
        BatchedMCTS mcts(board, half_komi, 1, device, 0, arena_slots, batch_size);
        if (!model_path.empty()) {
            mcts.load_model(model_path);
            mcts.set_agent(TZ_AGENT_NETWORK);
        }
        tz_state_t env = mcts.envs()[0];  // Env::default()
        if (!tps_text.empty() && !parse_tps(tps_text, board, &env)) throw std::runtime_error("--tps is not valid TPS");
        mcts.set_positions(std::vector<tz_state_t>(1, env));  // node = Node::default()
        auto terminal = [&]() {
            int t = 0;
            check(tz_result(mcts.handle(), &env, 1, &t));
            return t;
        };
        if (example) {  // run_example (main.rs:33-42)
            while (terminal() == 0) {
                std::cout << "tps: " << tps(env, board) << "\n";
                mcts.tree_simulate_batch(BETA, batch_size);
                const Move action = mcts.select_best_actions()[0];
                std::cout << ">>> " << move_to_string(action) << std::endl;
                mcts.tree_descend(action);
                env = mcts.envs()[0];
            }
            return 0;
        }
        std::string input;
        for (;;) {
            std::cout << "tps: " << tps(env, board) << "\n>>> " << std::flush;
            if (!std::getline(std::cin, input)) break;
            const size_t a = input.find_first_not_of(" \t\r\n"), b = input.find_last_not_of(" \t\r\n");
            const std::string trim = a == std::string::npos ? "" : input.substr(a, b - a + 1);
            Move mov;
            if (parse_move(trim, &mov)) {
                tz_state_t next = env;
                int ok = 0;
                check(tz_apply(mcts.handle(), &next, &mov, 1, &ok));
                if (!ok) {
                    std::cerr << "illegal move " << trim << "\n";  // `env.play` error: the position stays
                    continue;
                }
                mcts.tree_descend(mov);
                env = mcts.envs()[0];
            } else {
                mcts.tree_simulate_batch(BETA, batch_size);
            }
            std::cout << node_display(mcts) << "\n";  // println!("{node}"): Display ends with a newline already
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "analysis: %s\n", e.what());
        return 1;
    }
    return 0;
}
