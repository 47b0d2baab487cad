// takzero_b200.hpp -- C++17 host-side mirror of the reference's search surface on top of the C ABI
// (include/takzero_b200.h).  Header only; link against libtakzero_b200.so.
//
// The reference is Rust; its toolchain is not available where this was built, so the host layer that a
// `selfplay` / `reanalyze` style program needs is provided in C++ with the reference's names and semantics:
//   takzero::BatchedMCTS      takzero/src/search/node/batched.rs:24-409
//   takzero::Eval             takzero/src/search/eval.rs:8-163 (negate, f32::from; used for value targets)
//   takzero::Target / Replay  takzero/src/target.rs:25-30,56-73,167-170,215-232 (text formats of the files
//                             `learn` consumes), takzero::tps / move_to_string (takparse `Tps`, `Move` Display)
// All search / rules / network math happens in the CUDA library; this header only marshals and formats.
#pragma once

#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include "takzero_b200.h"

namespace takzero {

inline void check(int rc) {
    if (rc < 0) throw std::runtime_error(std::string(tz_last_error()) + " (code " + std::to_string(rc) + ")");
}

// ---- notation -----------------------------------------------------------------------------------------

using Move = tz_move_t;

// takparse `Move` Display: "a1", "Sa1", "Ca1", "a1+", "3a1>12" (drop counts omitted for a single drop)
inline std::string move_to_string(Move m) {
    std::string s;
    const int col = m & 7, row = (m >> 3) & 7, kind = (m >> 6) & 3, pat = m >> 8;
    if (pat == 0) {
        if (kind == 1) s += 'S';
        if (kind == 2) s += 'C';
        s += char('a' + col);
        s += char('1' + row);
        return s;
    }
    const int c = 8 - __builtin_ctz((unsigned)pat);
    if (c > 1) s += char('0' + c);
    s += char('a' + col);
    s += char('1' + row);
    s += "+-<>"[kind];
    int drops[8], nd = 0;
    for (int i = 0; i < c; i++) {
        if ((pat >> (8 - c + i)) & 1) drops[nd++] = 0;
        drops[nd - 1]++;
    }
    if (nd > 1)
        for (int i = 0; i < nd; i++) s += char('0' + drops[i]);
    return s;
}

// takparse `Tps` Display of a position: ranks from N down to 1, "x"/"xK" for empties, stacks bottom-up as
// 1/2 with S/C suffix, then the player to move (1/2) and the move number
inline std::string tps(const tz_state_t& g, int n) {
    std::string s;
    for (int row = n - 1; row >= 0; row--) {
        int empties = 0;
        bool first = true;
        for (int col = 0; col <= n; col++) {
            const int sq = row * n + col;
            if (col < n && g.height[sq] == 0) {
                empties++;
                continue;
            }
            if (empties) {
                if (!first) s += ',';
                s += 'x';
                if (empties > 1) s += char('0' + empties);
                empties = 0;
                first = false;
            }
            if (col == n) break;
            if (!first) s += ',';
            first = false;
            for (int i = 0; i < g.height[sq]; i++) s += char('1' + ((g.stack[sq] >> i) & 1));
            if (g.top[sq] == 1) s += 'S';
            if (g.top[sq] == 2) s += 'C';
        }
        if (row > 0) s += '/';
    }
    s += ' ';
    s += char('1' + g.to_move);
    s += ' ';
    s += std::to_string(g.ply / 2 + 1);
    return s;
}

// takparse `Move` FromStr (PTN): the inverse of move_to_string; returns false on malformed input
inline bool parse_move(const std::string& str, Move* out) {
    const char* s = str.c_str();
    int kind = 0, c = 0;
    if (*s == 'S') { kind = 1; s++; } else if (*s == 'C') { kind = 2; s++; } else if (*s == 'F') { s++; }
    if (*s >= '1' && *s <= '8') c = *s++ - '0';
    if (*s < 'a' || *s > 'h') return false;
    const int col = *s++ - 'a';
    if (*s < '1' || *s > '8') return false;
    const int row = *s++ - '1';
    if (*s == 0) {
        if (c != 0) return false;
        *out = (Move)(col | (row << 3) | (kind << 6));
        return true;
    }
    int dir;
    switch (*s++) {
        case '+': dir = 0; break;
        case '-': dir = 1; break;
        case '<': dir = 2; break;
        case '>': dir = 3; break;
        default: return false;
    }
    if (c == 0) c = 1;
    int drops[8], nd = 0, total = 0;
    while (*s >= '1' && *s <= '8' && nd < 8) {
        drops[nd] = *s++ - '0';
        total += drops[nd++];
    }
    while (*s == '*' || *s == '\'' || *s == '!' || *s == '?') s++;
    if (*s != 0) return false;
    if (nd == 0) { drops[nd++] = c; total = c; }
    if (total != c || c > 8) return false;
    int pat = 0, i = 0;
    for (int d = 0; d < nd; d++) {
        pat |= 1 << (8 - c + i);
        i += drops[d];
    }
    *out = (Move)(col | (row << 3) | (dir << 6) | (pat << 8));
    return true;
}

// takparse `Tps` FromStr into a tz_state_t (reserves are what is left of the standard piece counts;
// reversible_plies is not part of TPS and starts at 0, like `Game::from(tps)` in the reference)
inline bool parse_tps(const std::string& text, int n, tz_state_t* g) {
    static const int STONES[9] = {0, 0, 0, 10, 15, 21, 30, 40, 50}, CAPS[9] = {0, 0, 0, 0, 0, 1, 1, 2, 2};
    std::memset(g, 0, sizeof(*g));
    g->stones[0] = g->stones[1] = (uint8_t)STONES[n];
    g->caps[0] = g->caps[1] = (uint8_t)CAPS[n];
    const char* s = text.c_str();
    int row = n - 1, col = 0;
    while (*s && *s != ' ') {
        if (*s == '/') {
            if (col != n) return false;
            row--; col = 0; s++;
        } else if (*s == ',') {
            s++;
        } else if (*s == 'x') {
            s++;
            int k = 1;
            if (*s >= '1' && *s <= '8') k = *s++ - '0';
            col += k;
        } else if (*s == '1' || *s == '2') {
            if (row < 0 || col >= n) return false;
            const int sq = row * n + col;
            int h = 0;
            uint64_t bits = 0;
            while (*s == '1' || *s == '2') { bits |= (uint64_t)(*s - '1') << h; h++; s++; }
            int type = 0;
            if (*s == 'S') { type = 1; s++; } else if (*s == 'C') { type = 2; s++; }
            g->stack[sq] = bits;
            g->height[sq] = (uint8_t)h;
            g->top[sq] = (uint8_t)type;
            for (int i = 0; i < h; i++) {
                const int cl = (int)((bits >> i) & 1);
                uint8_t& pool = (i == h - 1 && type == 2) ? g->caps[cl] : g->stones[cl];
                if (pool == 0) return false;
                pool--;
            }
            col++;
        } else {
            return false;
        }
    }
    if (row != 0 || col != n) return false;
    int player = 1, move_no = 1;
    if (std::sscanf(s, " %d %d", &player, &move_no) != 2) return false;
    g->to_move = (uint8_t)(player - 1);
    g->ply = (uint16_t)((move_no - 1) * 2 + (player - 1));
    return true;
}

// Rust `{}` of an f32: the shortest decimal digits that round-trip, written positionally (never in
// exponent form): "1", "0.5", "-0.0009", "340000000000000000000000000000000000000"
inline std::string format_f32(float v) {
    if (std::isnan(v)) return "NaN";
    if (std::isinf(v)) return v > 0 ? "inf" : "-inf";
    if (v == 0.0f) return std::signbit(v) ? "-0" : "0";
    char buf[64];
    auto r = std::to_chars(buf, buf + sizeof(buf), std::fabs(v), std::chars_format::scientific);  // d.ddde[+-]XX
    std::string sci(buf, r.ptr);
    const size_t epos = sci.find('e');
    const int exp10 = std::atoi(sci.c_str() + epos + 1);
    std::string digits;
    for (size_t i = 0; i < epos; i++)
        if (sci[i] != '.') digits += sci[i];
    std::string out = std::signbit(v) ? "-" : "";
    const int point = exp10 + 1;  // position of the decimal point relative to the first digit
    if (point <= 0) {
        out += "0." + std::string((size_t)(-point), '0') + digits;
    } else if ((size_t)point >= digits.size()) {
        out += digits + std::string((size_t)point - digits.size(), '0');
    } else {
        out += digits.substr(0, (size_t)point) + "." + digits.substr((size_t)point);
    }
    return out;
}

inline const char* result_string(int game_result) {  // tz_game_result codes
    static const char* names[] = {"", "R-0", "0-R", "F-0", "0-F", "1/2-1/2"};
    return names[game_result];
}

// ---- Eval (search/eval.rs) ------------------------------------------------------------------------------

struct Eval {
    uint32_t tag = 0;  // 0 Value, 1 Win, 2 Loss, 3 Draw
    union {
        float value;
        uint32_t ply;
    };
    Eval() : value(0.0f) {}
    static Eval from_terminal(int terminal) {  // eval.rs:118-126; terminal: 1 win, 2 loss, 3 draw
        Eval e;
        e.tag = (uint32_t)terminal;
        e.ply = 0;
        return e;
    }
    Eval negate() const {  // eval.rs:40-47
        Eval e = *this;
        switch (tag) {
            case 0: e.value = -value; break;
            case 1: e.tag = 2; e.ply = ply + 1; break;
            case 2: e.tag = 1; e.ply = ply + 1; break;
            default: e.ply = ply + 1; break;
        }
        return e;
    }
    float to_f32() const {  // eval.rs:95-105, `0.997f32.powi(ply)` by square-and-multiply like compiler-rt
        if (tag == 0) return value;
        float a = 0.997f, r = 1.0f;
        for (uint32_t b = ply;;) {
            if (b & 1) r *= a;
            b >>= 1;
            if (b == 0) break;
            a *= a;
        }
        return r * (tag == 1 ? 1.0f : tag == 2 ? -1.0f : 0.0f);
    }
};

// ---- Target / Replay (target.rs) ---------------------------------------------------------------------------

struct Target {
    tz_state_t env;
    std::vector<std::pair<Move, float>> policy;
    float value = 0.0f;
    float ube = 0.0f;
    // "{tps};{value};{ube};{move:p,move:p,...}\n" (target.rs:56-73)
    std::string to_string(int n) const {
        std::string s = tps(env, n) + ';' + format_f32(value) + ';' + format_f32(ube) + ';';
        for (size_t i = 0; i < policy.size(); i++) {
            if (i) s += ',';
            s += move_to_string(policy[i].first) + ':' + format_f32(policy[i].second);
        }
        s += '\n';
        return s;
    }
    // Target FromStr (target.rs:98-140) up to the check against the position's legal moves (that needs the rules,
    // i.e. tz_legal_moves; callers with a handle do it): "{tps};{value};{ube};{move:p,...}"
    static bool parse(const std::string& line, int n, Target* out) {
        std::string s = line;
        while (!s.empty() && (s.back() == '\n' || s.back() == '\r' || s.back() == ' ')) s.pop_back();
        std::vector<std::string> parts;
        for (size_t pos = 0;;) {
            const size_t end = s.find(';', pos);
            parts.push_back(s.substr(pos, end == std::string::npos ? std::string::npos : end - pos));
            if (end == std::string::npos) break;
            pos = end + 1;
        }
        if (parts.size() < 4) return false;  // MissingTps / MissingValue / MissingUbe / MissingPolicy
        if (!parse_tps(parts[0], n, &out->env)) return false;
        auto parse_float = [](const std::string& t, float* v) {
            if (t.empty()) return false;
            char* end = nullptr;
            *v = std::strtof(t.c_str(), &end);
            return end == t.c_str() + t.size();
        };
        if (!parse_float(parts[1], &out->value) || !parse_float(parts[2], &out->ube)) return false;
        out->policy.clear();
        for (size_t pos = 0; pos <= parts[3].size();) {
            size_t end = parts[3].find(',', pos);
            if (end == std::string::npos) end = parts[3].size();
            const std::string item = parts[3].substr(pos, end - pos);
            const size_t colon = item.find(':');
            if (colon == std::string::npos) return false;  // WrongPolicyFormat
            Move m;
            float p;
            if (!parse_move(item.substr(0, colon), &m) || !parse_float(item.substr(colon + 1), &p) || std::isnan(p))
                return false;
            out->policy.emplace_back(m, p);
            pos = end + 1;
        }
        return true;
    }
};

struct Replay {
    tz_state_t env;
    std::vector<Move> actions;
    // "[TPS \"{tps}\"] m1 m2 ... {result}\n" (target.rs:215-232); game_result from tz_game_result (0 = none)
    std::string to_string(int n, int game_result) const {
        std::string s = "[TPS \"" + tps(env, n) + "\"]";
        for (Move m : actions) s += ' ' + move_to_string(m);
        if (game_result) s += std::string(" ") + result_string(game_result);
        s += '\n';
        return s;
    }
    // Replay FromStr (target.rs:243-272): `[TPS "..."] m1 m2 ... [result]`
    static bool parse(const std::string& line, int n, Replay* out) {
        const size_t a = line.find('"'), b = line.find('"', a + 1);
        if (a == std::string::npos || b == std::string::npos) return false;
        if (!parse_tps(line.substr(a + 1, b - a - 1), n, &out->env)) return false;
        out->actions.clear();
        size_t pos = line.find(']', b);
        if (pos == std::string::npos) return false;
        pos++;
        while (pos < line.size()) {
            while (pos < line.size() && line[pos] == ' ') pos++;
            size_t end = line.find(' ', pos);
            if (end == std::string::npos) end = line.size();
            const std::string tok = line.substr(pos, end - pos);
            pos = end;
            if (tok.empty()) continue;
            Move m;
            if (parse_move(tok, &m)) out->actions.push_back(m);
            else if (tok.find('-') == std::string::npos) return false;  // not a result token either
        }
        return true;
    }
};

// ---- files the reference's processes synchronise through ------------------------------------------------------

// `buffer_lengths.txt`, written by learn/src/main.rs:195-209 as "{selfplay},{reanalyze},{sum}" and read by
// read_buffer_lengths (selfplay/src/main.rs:371-387, reanalyze/src/main.rs:304-320): status 0 ok, -1 no such file
// (io error), -2 missing component / wrong checksum (torn read)
struct BufferLengths {
    int status = -1;
    size_t selfplay = 0, reanalyze = 0;
};
inline BufferLengths read_buffer_lengths(const std::string& directory) {
    BufferLengths out;
    std::ifstream f(directory + "/buffer_lengths.txt");
    if (!f) return out;
    const std::string text((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    std::vector<unsigned long long> nums;
    std::stringstream ss(text);
    std::string tok;
    while (std::getline(ss, tok, ',')) {
        char* end = nullptr;
        const unsigned long long v = std::strtoull(tok.c_str(), &end, 10);
        if (end != tok.c_str() && (*end == 0 || *end == '\n')) nums.push_back(v);
    }
    out.status = -2;
    if (nums.size() < 3 || nums[0] + nums[1] != nums[2]) return out;
    out.status = 0;
    out.selfplay = (size_t)nums[0];
    out.reanalyze = (size_t)nums[1];
    return out;
}

// Appends `contents` with ONE write() on an O_APPEND descriptor, so that several processes (one per GPU) can share
// `targets-*.txt` / `replays.txt` without tearing each other's lines (save_targets_to_file, selfplay/src/main.rs:
// 332-346).  Returns false when the file cannot be written.
inline bool append_file(const std::string& path, const std::string& contents) {
    const int fd = ::open(path.c_str(), O_WRONLY | O_CREAT | O_APPEND, 0644);
    if (fd < 0) return false;
    size_t done = 0;
    while (done < contents.size()) {
        const ssize_t n = ::write(fd, contents.data() + done, contents.size() - done);
        if (n <= 0) break;
        done += (size_t)n;
    }
    ::close(fd);
    return done == contents.size();
}

inline long long mtime_ns(const std::string& path) {
    struct stat st;
    if (stat(path.c_str(), &st) != 0) return -1;
    return (long long)st.st_mtim.tv_sec * 1000000000LL + st.st_mtim.tv_nsec;
}

// ---- model files: the reference's `model_latest.ot` (tch VarStore archive), a `torch.save` state dict or this
// repository's TZW1 container, all parsed by the library (tz_read_model_file) -----------------------------------

struct Weights {
    std::vector<std::string> names;
    std::vector<std::vector<int64_t>> shapes;
    std::vector<std::vector<float>> data;
    static Weights load(const std::string& path) {  // Tensor::load_multi
        Weights w;
        check(tz_read_model_file(
            path.c_str(),
            [](void* ctx, const char* name, const char*, const float* data, const int64_t* shape, int ndim) {
                Weights& self = *static_cast<Weights*>(ctx);
                self.names.emplace_back(name);
                self.shapes.emplace_back(shape, shape + ndim);
                size_t numel = 1;
                for (int i = 0; i < ndim; i++) numel *= (size_t)shape[i];
                self.data.emplace_back(data, data + numel);
            },
            &w));
        return w;
    }
};

// ---- BatchedMCTS (search/node/batched.rs) --------------------------------------------------------------------

class BatchedMCTS {
  public:
    BatchedMCTS(int board_n, int half_komi, int n_games, int device = 0, int game_base = 0, uint32_t arena_slots = 0,
                int tree_batch = 0)
        : n_(board_n), games_(n_games) {
        tz_config_t cfg{};
        cfg.board_n = board_n;
        cfg.half_komi = half_komi;
        cfg.n_games = n_games;
        cfg.device = device;
        cfg.game_base = game_base;
        cfg.arena_slots = arena_slots;
        cfg.tree_batch = tree_batch;
        check(tz_create(&cfg, &h_));
        check(tz_info(h_, &stride_, nullptr, nullptr, nullptr));
    }
    ~BatchedMCTS() { tz_destroy(h_); }
    BatchedMCTS(const BatchedMCTS&) = delete;
    BatchedMCTS& operator=(const BatchedMCTS&) = delete;

    tz_handle* handle() const { return h_; }
    int board_n() const { return n_; }
    int games() const { return games_; }
    int move_stride() const { return stride_; }

    void set_weights(const Weights& w) {  // Net::load
        std::vector<tz_tensor_t> t(w.names.size());
        for (size_t i = 0; i < t.size(); i++)
            t[i] = tz_tensor_t{w.names[i].c_str(), w.data[i].data(), w.shapes[i].data(), (int)w.shapes[i].size()};
        check(tz_set_weights(h_, t.data(), (int)t.size()));
    }
    // Net::load(path, device) (network/mod.rs:20-27, net6_simhash.rs:164-181) incl. the `bitvec.bin` sidecar
    void load_model(const std::string& path) { check(tz_load_model(h_, path.c_str())); }
    // ---- several GPUs, one process each (csrc/comm.cu): NCCL communicator, weight generations, counter sums ----------
    static std::vector<uint8_t> comm_unique_id() {  // by one rank; the 128 bytes reach the others by the host's own means
        std::vector<uint8_t> id(128);
        check(tz_comm_unique_id(id.data()));
        return id;
    }
    void comm_init(const std::vector<uint8_t>& id, int nranks, int rank) {
        check(tz_comm_init(h_, nranks > 1 ? id.data() : nullptr, nranks, rank));
    }
    // The per-move `Net::load` of selfplay/src/main.rs:107 as ONE collective: the root passes the model, the others
    // nullptr (and the number of residual blocks, 0 = the board's default); all ranks swap weight sets between moves.
    void broadcast_weights(const Weights* w, int root = 0, int res_blocks = 0) {
        if (!w) {
            check(tz_broadcast_weights(h_, nullptr, 0, res_blocks, root));
            return;
        }
        std::vector<tz_tensor_t> t(w->names.size());
        for (size_t i = 0; i < t.size(); i++)
            t[i] = tz_tensor_t{w->names[i].c_str(), w->data[i].data(), w->shapes[i].data(), (int)w->shapes[i].size()};
        check(tz_broadcast_weights(h_, t.data(), (int)t.size(), res_blocks, root));
    }
    std::vector<uint64_t> allreduce_sum(std::vector<uint64_t> values) {
        check(tz_allreduce_sum(h_, values.data(), (int)values.size()));
        return values;
    }
    // ---- reanalyze on the device (reanalyze/src/main.rs:147-235) -------------------------------------------------------
    void stage_positions(const std::vector<tz_state_t>& buffer) { check(tz_stage_positions(h_, buffer.data(), buffer.size())); }
    void reanalyze_batch(const std::vector<uint32_t>* pool_indices, int sampled_actions, uint32_t budget, float ube_beta,
                         uint64_t seed) {
        const tz_reanalyze_t p{sampled_actions, budget, ube_beta, seed};
        check(tz_reanalyze_batch(h_, pool_indices ? pool_indices->data() : nullptr, &p));
    }
    struct ReanalyzeTargets {
        std::vector<float> policy, ube, value;
        std::vector<int> n;
        std::vector<Move> moves;
    };
    ReanalyzeTargets reanalyze_read() {
        ReanalyzeTargets t;
        const size_t cells = (size_t)games_ * stride_;
        t.policy.resize(cells);
        t.moves.resize(cells);
        t.ube.resize(games_);
        t.value.resize(games_);
        t.n.resize(games_);
        check(tz_reanalyze_read(h_, stride_, t.policy.data(), t.ube.data(), t.value.data(), t.n.data(), t.moves.data()));
        return t;
    }
    // ---- resident self-play (selfplay/src/main.rs:138-153,238-329 on the device) ----------------------------------------
    // one whole move of every game, asynchronous; with recording on, its training data stays on the device
    void selfplay_move(const tz_selfplay_t& params) { check(tz_selfplay_move(h_, &params)); }
    void selfplay_record(bool enable, size_t bytes_per_game = 0, size_t output_bytes = 0) {
        check(tz_selfplay_record(h_, enable ? 1 : 0, bytes_per_game, output_bytes));
    }
    struct FinishedGame {
        Replay replay;
        int result = 0;     // tz_game_result code of the final position
        int terminal = 0;   // tz_result code of the final position
        int game = 0;       // global game id
        bool exploration = false;
    };
    struct SelfplayData {
        std::vector<Target> targets;  // finished games in ascending order, each from its last ply to its first
        std::vector<int> target_games;
        std::vector<FinishedGame> games;
        size_t high_water_bytes = 0;
    };
    // completed targets and finished replays since the last read (waits for the device, empties the queue)
    SelfplayData selfplay_read() {
        tz_selfplay_data_t io{};
        const int rc = tz_selfplay_read(h_, &io);  // capacities 0: the counts
        if (rc != TZ_EINVAL || (io.n_targets | io.n_policy | io.n_replays | io.n_moves) == 0) check(rc);
        std::vector<tz_state_t> t_env(io.n_targets), r_start(io.n_replays);
        std::vector<float> t_value(io.n_targets), t_ube(io.n_targets), probs(io.n_policy);
        std::vector<int> t_n(io.n_targets), t_game(io.n_targets), r_result(io.n_replays), r_term(io.n_replays),
            r_len(io.n_replays), r_game(io.n_replays);
        std::vector<uint64_t> t_off(io.n_targets), r_off(io.n_replays);
        std::vector<Move> moves(io.n_policy), r_moves(io.n_moves);
        std::vector<uint8_t> r_expl(io.n_replays);
        if (rc != TZ_OK) {
            io.target_cap = io.n_targets;
            io.policy_cap = io.n_policy;
            io.replay_cap = io.n_replays;
            io.move_cap = io.n_moves;
            io.target_env = t_env.data();
            io.target_value = t_value.data();
            io.target_ube = t_ube.data();
            io.target_n = t_n.data();
            io.target_offset = t_off.data();
            io.target_game = t_game.data();
            io.policy_moves = moves.data();
            io.policy_probs = probs.data();
            io.replay_start = r_start.data();
            io.replay_result = r_result.data();
            io.replay_terminal = r_term.data();
            io.replay_length = r_len.data();
            io.replay_offset = r_off.data();
            io.replay_game = r_game.data();
            io.replay_exploration = r_expl.data();
            io.replay_moves = r_moves.data();
            check(tz_selfplay_read(h_, &io));
        }
        SelfplayData out;
        out.high_water_bytes = io.high_water_bytes;
        out.targets.resize(io.n_targets);
        out.target_games = t_game;
        for (size_t i = 0; i < io.n_targets; i++) {
            Target& t = out.targets[i];
            t.env = t_env[i];
            t.value = t_value[i];
            t.ube = t_ube[i];
            t.policy.reserve((size_t)t_n[i]);
            for (int j = 0; j < t_n[i]; j++) t.policy.emplace_back(moves[t_off[i] + j], probs[t_off[i] + j]);
        }
        out.games.resize(io.n_replays);
        for (size_t i = 0; i < io.n_replays; i++) {
            FinishedGame& f = out.games[i];
            f.replay.env = r_start[i];
            f.replay.actions.assign(r_moves.begin() + (ptrdiff_t)r_off[i], r_moves.begin() + (ptrdiff_t)(r_off[i] + r_len[i]));
            f.result = r_result[i];
            f.terminal = r_term[i];
            f.game = r_game[i];
            f.exploration = r_expl[i] != 0;
        }
        return out;
    }
    void set_agent(int kind, tz_agent_fn fn = nullptr, void* ctx = nullptr) { check(tz_set_agent(h_, kind, fn, ctx)); }
    void new_openings(uint64_t seed) { check(tz_new_openings(h_, nullptr, nullptr, nullptr, seed)); }
    void set_positions(const std::vector<tz_state_t>& envs) { check(tz_set_positions(h_, envs.data(), nullptr)); }
    // only the games with mask[g] != 0: `*node = Node::default(); *env = envs[g]`
    void set_positions(const std::vector<tz_state_t>& envs, const std::vector<uint8_t>& mask) {
        check(tz_set_positions(h_, envs.data(), mask.data()));
    }
    // the random part of Env::new_opening_with_random_steps (env.rs:81-96) for the masked games (all: empty mask)
    void random_steps(int steps, uint64_t seed, const std::vector<uint8_t>& mask = {}) {
        check(tz_random_steps(h_, mask.empty() ? nullptr : mask.data(), steps, seed));
    }
    std::vector<tz_state_t> envs() const {
        std::vector<tz_state_t> out(games_);
        check(tz_get_positions(h_, out.data()));
        return out;
    }
    void simulate(const std::vector<float>& betas) { check(tz_simulate(h_, betas.data())); }
    // noise drawn by the library from `seed` (the reference draws from its rng, whose stream is not pinned)
    std::vector<Move> gumbel_sequential_halving(const std::vector<float>& betas, int sampled_actions,
                                                uint32_t search_budget, uint64_t seed) {
        std::vector<Move> out(games_);
        check(tz_gumbel_sequential_halving(h_, betas.data(), sampled_actions, search_budget, nullptr, 0, seed, out.data()));
        return out;
    }
    std::vector<Move> select_actions_in_selfplay(int weighted_random_plies, uint64_t seed, uint32_t threshold = 32,
                                                 float allowed_eval_drop = 0.5f) {
        std::vector<Move> out(games_);
        check(tz_select_selfplay(h_, weighted_random_plies, threshold, allowed_eval_drop, nullptr, seed, out.data()));
        return out;
    }
    std::vector<Move> select_best_actions() {
        std::vector<Move> out(games_);
        check(tz_select_best(h_, out.data()));
        return out;
    }
    void step(const std::vector<Move>& actions) { check(tz_step(h_, actions.data())); }
    // Replay::states (target.rs:205-212) of many replays at once: the position before every action, replay by
    // replay in file order.  The moves are applied on the device, all replays in lock-step by ply (one tz_apply per
    // ply index instead of one per position).
    std::vector<tz_state_t> replay_states(const std::vector<Replay>& replays) {
        std::vector<size_t> first(replays.size() + 1, 0);
        size_t longest = 0;
        for (size_t r = 0; r < replays.size(); r++) {
            first[r + 1] = first[r] + replays[r].actions.size();
            longest = std::max(longest, replays[r].actions.size());
        }
        std::vector<tz_state_t> out(first.back());
        std::vector<tz_state_t> cur;
        std::vector<size_t> who;
        for (size_t r = 0; r < replays.size(); r++)
            if (!replays[r].actions.empty()) {
                who.push_back(r);
                cur.push_back(replays[r].env);
            }
        std::vector<Move> moves;
        std::vector<int> ok;
        for (size_t ply = 0; ply < longest && !who.empty(); ply++) {
            moves.resize(who.size());
            ok.assign(who.size(), 0);
            for (size_t i = 0; i < who.size(); i++) {
                out[first[who[i]] + ply] = cur[i];
                moves[i] = replays[who[i]].actions[ply];
            }
            check(tz_apply(h_, cur.data(), moves.data(), (int)who.size(), ok.data()));
            size_t keep = 0;
            for (size_t i = 0; i < who.size(); i++) {
                if (!ok[i]) throw std::runtime_error("Action should be valid: " + move_to_string(moves[i]));
                if (ply + 1 < replays[who[i]].actions.size()) {
                    who[keep] = who[i];
                    cur[keep] = cur[i];
                    keep++;
                }
            }
            who.resize(keep);
            cur.resize(keep);
        }
        return out;
    }
    std::vector<tz_state_t> replay_states(const Replay& r) { return replay_states(std::vector<Replay>(1, r)); }

    struct RootTargets {
        std::vector<float> policy;  // [games][stride]
        std::vector<Move> moves;    // [games][stride]
        std::vector<int> n;
        std::vector<float> ube;
    };
    // Node::improved_policy + Node::ube_target of every root (visitations < 0: most_visited_count())
    RootTargets targets(float visitations, float beta) {
        RootTargets t;
        t.policy.resize((size_t)games_ * stride_);
        t.moves.resize((size_t)games_ * stride_);
        t.n.resize(games_);
        t.ube.resize(games_);
        check(tz_targets(h_, visitations, beta, stride_, t.policy.data(), t.ube.data(), t.n.data(), t.moves.data()));
        return t;
    }
    struct RootStats {
        std::vector<tz_root_t> roots;
    };
    std::vector<tz_root_t> root_stats() {
        std::vector<tz_root_t> out(games_);
        check(tz_root_stats(h_, out.data()));
        return out;
    }
    struct Children {
        int stride;
        std::vector<int> n;
        std::vector<Move> moves;
        std::vector<uint32_t> visits, eval_tag, eval_bits;
        std::vector<float> logit, prob, std_dev;
    };
    Children root_children() {
        Children c;
        c.stride = stride_;
        const size_t cells = (size_t)games_ * stride_;
        c.n.resize(games_);
        c.moves.resize(cells);
        c.visits.resize(cells);
        c.eval_tag.resize(cells);
        c.eval_bits.resize(cells);
        c.logit.resize(cells);
        c.prob.resize(cells);
        c.std_dev.resize(cells);
        check(tz_root_children(h_, stride_, c.n.data(), c.moves.data(), c.visits.data(), c.eval_tag.data(),
                               c.eval_bits.data(), c.logit.data(), c.prob.data(), c.std_dev.data()));
        return c;
    }
    // restart_terminal_envs: terminal[g] (0 none, 1 win, 2 loss, 3 draw for the side to move) and, for finished
    // games, the replay that just ended
    std::vector<int> restart_terminal_envs(uint64_t seed) {
        std::vector<int> term(games_);
        check(tz_restart_terminal(h_, nullptr, nullptr, seed, term.data()));
        return term;
    }
    Replay finished_replay(int game) {
        Replay r;
        std::vector<Move> buf(TZ_MAX_PLIES);
        const int len = tz_finished_replay(h_, game, &r.env, buf.data(), TZ_MAX_PLIES);
        check(len);
        r.actions.assign(buf.begin(), buf.begin() + len);
        return r;
    }
    // ---- single tree = game 0 (tei / analysis): Node::simulate_simple / simulate_batch / descend / PV ----
    void tree_simulate_simple(float beta) { check(tz_tree_simulate_simple(h_, beta)); }
    void tree_simulate_batch(float beta, int batch_size) { check(tz_tree_simulate_batch(h_, beta, batch_size)); }
    void tree_descend(Move m) { check(tz_tree_descend(h_, m)); }
    std::vector<Move> principal_variation(int cap = 64) {
        std::vector<Move> pv(cap);
        const int len = tz_tree_principal_variation(h_, pv.data(), cap);
        check(len);
        pv.resize(len);
        return pv;
    }
    // ---- many single trees at once: the tree of every game with mask[g] != 0 (all: empty mask) ----
    void trees_simulate_batch(float beta, int batch_size, const std::vector<uint8_t>& mask = {}) {
        check(tz_trees_simulate_batch(h_, mask.empty() ? nullptr : mask.data(), beta, batch_size));
    }
    // moves [n_games]; unselected games' entries are ignored
    void trees_descend(const std::vector<Move>& moves, const std::vector<uint8_t>& mask = {}) {
        check(tz_trees_descend(h_, mask.empty() ? nullptr : mask.data(), moves.data()));
    }
    // one principal variation per game (empty for unselected games)
    std::vector<std::vector<Move>> trees_principal_variation(int cap = 64, const std::vector<uint8_t>& mask = {}) {
        std::vector<Move> buf((size_t)games_ * cap);
        std::vector<int> len(games_);
        check(tz_trees_principal_variation(h_, mask.empty() ? nullptr : mask.data(), cap, buf.data(), len.data()));
        std::vector<std::vector<Move>> pv(games_);
        for (int g = 0; g < games_; g++) pv[g].assign(buf.begin() + (size_t)g * cap, buf.begin() + (size_t)g * cap + len[g]);
        return pv;
    }
    tz_counters_t counters() {
        tz_counters_t c;
        check(tz_counters(h_, &c));
        return c;
    }

  private:
    tz_handle* h_ = nullptr;
    int n_, games_, stride_ = 0;
};

// ---- `impl Display for Node` (search/node/debug.rs:11-95): the table the `analysis` REPL prints -------------------

inline std::string center(const std::string& s, size_t width) {  // Rust `{: ^width}`: the odd space goes right
    if (s.size() >= width) return s;
    const size_t pad = width - s.size(), left = pad / 2;
    return std::string(left, ' ') + s + std::string(pad - left, ' ');
}
inline std::string fixed4(float v, bool plus) {  // `{:.4}` / `{:+.4}` of an f32
    char buf[64];
    std::snprintf(buf, sizeof(buf), plus ? "%+.4f" : "%.4f", (double)v);
    return buf;
}
inline std::string eval_display(uint32_t tag, uint32_t bits) {  // `{:+.4}` of an Eval (eval.rs:15-24)
    if (tag == 0) {
        float v;
        std::memcpy(&v, &bits, 4);
        return fixed4(v, true);
    }
    return std::string(tag == 1 ? "Win(" : tag == 2 ? "Loss(" : "Draw(") + std::to_string(bits) + ")";
}
// game `g` of the handle: children sorted by visit count (stable), one `ActionInfo` row each, header, node line
inline std::string node_display(BatchedMCTS& mcts, int g = 0) {
    const BatchedMCTS::Children ch = mcts.root_children();
    const std::vector<tz_root_t> roots = mcts.root_stats();
    const tz_root_t& root = roots[g];
    std::string out;
    float std_dev;
    std::memcpy(&std_dev, &root.std_dev_bits, 4);
    const size_t base = (size_t)g * ch.stride;
    const int n = ch.n[g];
    if (n == 0 && root.eval_tag == 0) {  // needs_initialization: no children and not known
        out += "--- This node still needs to be initialized! ---\n";
    } else {
        const BatchedMCTS::RootTargets rt = mcts.targets(-1.0f, 0.0f);  // improved_policy(most_visited_count())
        std::vector<int> order(n);
        for (int i = 0; i < n; i++) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return ch.visits[base + a] < ch.visits[base + b]; });
        const float parent = (float)root.visit_count;
        // exploration_rate(N) * P * sqrt(N) / (1 + n)   (policy.rs:143-156)
        const float rate = std::log((1.0f + parent + 500.0f) / 500.0f) + 4.0f;
        for (int i : order) {
            const float puct = rate * ch.prob[base + i] * std::sqrt(parent) / (1.0f + (float)ch.visits[base + i]);
            out += center(move_to_string(ch.moves[base + i]), 10) + ' ' + center(std::to_string(ch.visits[base + i]), 9) + ' ' +
                   center(fixed4(ch.logit[base + i], true), 9) + ' ' + center(fixed4(ch.prob[base + i], false), 9) + ' ' +
                   center(fixed4(rt.policy[base + i], false), 9) + ' ' + center(fixed4(puct, false), 8) + ' ' +
                   center(fixed4(ch.std_dev[base + i], false), 9) + ' ' +
                   center(eval_display(ch.eval_tag[base + i], ch.eval_bits[base + i]), 14) + '\n';
        }
        out += "[ action ] [ count ] [ logit ] [ proba ] [ impol ] [ puct ] [ stdev ] [ evaluation ]\n";
    }
    out += "((node))  [count: " + std::to_string(root.visit_count) + "]  [std_dev: " + fixed4(std_dev, false) +
           "]  [eval: " + eval_display(root.eval_tag, root.eval_bits) + "]\n";
    return out;
}

}  // namespace takzero
