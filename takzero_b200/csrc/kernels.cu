// kernels.cu -- warp-per-game rules / tree kernels of the batched self-play search (sm_100a).
//
// One warp owns one game for the whole kernel: the position lives in shared memory
// (TzState, 384 B), the tree in the game's struct-of-arrays arena in HBM (children of a
// node are contiguous, so a warp reads 32 children per 128-byte transaction).
// What each kernel replaces in the reference (paths relative to takzero/src/):
//   k_select        search/node/mcts.rs:107-163 (forward, backward_known_eval) as driven by
//                   search/node/batched.rs:63-100,254-295; env.rs:39-59 (fast-tak rules)
//   k_expand        node/policy.rs:10-19 (softmax), mcts.rs:171-225 (backward_network_eval)
//   k_gumbel_init   batched.rs:226-244      k_halve     batched.rs:338-355
//   k_finalize      batched.rs:358-406      k_step      batched.rs:131-144, node/mod.rs:95-102
//   k_restart       batched.rs:185-203, env.rs:65-79
//   k_targets       node/policy.rs:23-48, node/mod.rs:215-230
//   k_select_actions node/mod.rs:132-207
#include "encode.cuh"
#include "kernels.cuh"
#include "rules.cuh"
#include "tree.cuh"

#define WPB TZ_WARPS_PER_BLOCK

__device__ __forceinline__ void flag_error(const TzDev& d, uint32_t bit, int lane) {
    if (lane == 0) atomicOr(d.status, bit);
}

__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }

// ---- one lock-step simulation: selection -----------------------------------------

// Node::forward (mcts.rs:107-138) from node `slot` with the position in `st` (shared memory):
// visit counts are incremented on the way down, the path is written to `traj`.
// Returns 1 when the result is known (*known_ev), 0 when the leaf needs the network, -1 on error.
__device__ __forceinline__ int warp_forward(const TzDev& d, const GameTree& t, TzState* st, uint32_t* traj,
                                            uint32_t slot, float beta, int lane, int* out_len, Ev* known_ev) {
    int len = 0;
    while (true) {
        if (len >= TZ_MAX_DEPTH) {
            flag_error(d, TZ_ERR_DEPTH, lane);
            return -1;
        }
        if (lane == 0) {
            t.visits[slot] += 1;
            traj[len] = slot;
        }
        len++;
        __syncwarp();
        const uint32_t meta = t.meta[slot];
        const uint32_t tag = tz_meta_tag(meta);
        if (tag != TZ_E_VALUE && t.eval[slot] == 0) {  // is_terminal
            *known_ev = ev_make(tag, 0);
            *out_len = len;
            return 1;
        }
        if (tz_meta_nchild(meta) == 0 && tag == TZ_E_VALUE) {  // needs_initialization
            const int term = warp_terminal(st, d.n, d.half_komi, d.rev_limit, lane);
            *out_len = len;
            if (term != TZ_T_NONE) {
                *known_ev = ev_make(term == TZ_T_WIN ? TZ_E_WIN : (term == TZ_T_LOSS ? TZ_E_LOSS : TZ_E_DRAW), 0);
                if (lane == 0) {
                    node_set_eval(t, slot, *known_ev);
                    t.std_dev[slot] = 0.0f;
                }
                __syncwarp();
                return 1;
            }
            return 0;
        }
        bool nan_seen;
        const int idx = warp_select_puct(t, slot, beta, d.ln_table, lane, &nan_seen);
        if (nan_seen) flag_error(d, TZ_ERR_NAN, lane);
        if (idx < 0) {
            flag_error(d, TZ_ERR_NO_CHILD, lane);
            return -1;
        }
        slot = t.first[slot] + (uint32_t)idx;
        if (!warp_apply(st, d.n, (uint16_t)tz_meta_move(t.meta[slot]), lane)) flag_error(d, TZ_ERR_BAD_MOVE, lane);
    }
}

// Forward::NeedsNetwork: legal moves + leaf position into evaluation-queue slot q
__device__ __forceinline__ bool warp_enqueue(const TzDev& d, int g, int q, TzState* st, uint16_t* moves, int lane) {
    const int cnt = warp_movegen(st, d.n, moves, lane, d.sq_ranges + (size_t)q * TZ_MAX_SQ);
    if (cnt < 0 || cnt > d.M) {
        // reported, never truncated; the queue slot is already taken, so it is filled with a well-formed entry without
        // moves (the agent and k_expand then have nothing to read out of bounds)
        flag_error(d, TZ_ERR_TOO_MANY_MOVES, lane);
        if (lane == 0) {
            d.nn_queue[q] = g;
            d.n_actions[q] = 0;
        }
        for (int sq = lane; sq < TZ_MAX_SQ; sq += 32) d.sq_ranges[(size_t)q * TZ_MAX_SQ + sq] = 0;
        warp_store_state(&d.leaf_state[q], st, lane);
        return false;
    }
    // what the network's input encoding needs of the whole position rides along in the queued copy: the flat count
    // difference and the six scalar planes (network/repr.rs:199-227)
    const TzBoards b = warp_boards(st, d.nn, lane);
    if (lane == 0) {
        d.nn_queue[q] = g;
        d.n_actions[q] = cnt;
        enc::store_position_scalars(st, __popcll(b.flat[0]) - __popcll(b.flat[1]), d.n, d.half_komi, d.nn_f16);
    }
    __syncwarp();
    warp_store_state(&d.leaf_state[q], st, lane);
    uint16_t* out = d.actions + (size_t)q * d.M;
    for (int i = lane; i < cnt; i += 32) out[i] = moves[i];
    return true;
}

__global__ void __launch_bounds__(32 * WPB) k_select(TzDev d, int phase, int halving_i, const float* betas) {
    __shared__ TzState s_state[WPB];
    __shared__ uint16_t s_moves[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    TzState* st = &s_state[warp];
    warp_load_state(st, &d.env[g], lane);
    const GameTree t = game_tree(d.arena, g);
    uint32_t* traj = d.traj + (size_t)g * TZ_MAX_DEPTH;
    unsigned long long* ctr = d.counters + (size_t)g * 4;

    uint32_t slot = 0;
    float beta = 0.0f;
    if (phase == 0) {
        beta = betas ? betas[g] : 0.0f;
    } else {
        // batched.rs:255-264: simulate below the i-th surviving root child (index wraps)
        const int len = d.set_len[g];
        if (len <= 0) {
            flag_error(d, TZ_ERR_SET_EMPTY, lane);
            return;
        }
        const int child = d.set_child[(size_t)g * TZ_MAX_K + (halving_i % len)];
        slot = t.first[0] + (uint32_t)child;
        if (!warp_apply(st, d.n, (uint16_t)tz_meta_move(t.meta[slot]), lane)) flag_error(d, TZ_ERR_BAD_MOVE, lane);
    }
    if (lane == 0) ctr[0] += 1;
    int len = 0;
    Ev known_ev = ev_value(0.0f);
    const int res = warp_forward(d, t, st, traj, slot, beta, lane, &len, &known_ev);
    if (res < 0) return;
    if (res == 1) {
        if (lane == 0) ctr[2] += 1;
        Propagated p;
        p.eval = known_ev;
        p.variance = 0.0f;
        warp_backup(t, traj, len, p, lane);
        return;
    }
    int q = 0;
    if (lane == 0) {
        q = atomicAdd(d.nn_count, 1);
        d.traj_len[g] = len;
        ctr[1] += 1;
    }
    q = __shfl_sync(FULL_MASK, q, 0);
    warp_enqueue(d, g, q, st, s_moves[warp], lane);
}

// ---- synthetic agent (oracle/tak_search.c `tk_agent_synthetic`) ----------------------

__global__ void __launch_bounds__(32 * WPB) k_agent_synth(TzDev d) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WPB + warp;
    if (q >= *d.nn_count) return;
    const uint64_t h = warp_state_hash(&d.leaf_state[q], d.nn, lane);
    const int cnt = d.n_actions[q];
    const uint16_t* act = d.actions + (size_t)q * d.M;
    float* lg = d.logits + (size_t)q * d.M;
    for (int i = lane; i < cnt; i += 32) {
        const uint64_t hm = tz_mix64(h ^ ((uint64_t)act[i] * 0x9e3779b97f4a7c15ULL));
        lg[i] = (float)((int)(hm & 0x7fff) - 16384) * (1.0f / 4096.0f);
    }
    if (lane == 0) {
        d.value[q] = (float)((int)((h >> 20) & 0xffff) - 32768) * (0.75f / 32768.0f);
        d.variance[q] = (float)((h >> 40) & 0xffff) * (1.0f / 65536.0f);
    }
}

// ---- one lock-step simulation: softmax + expansion + backup ------------------------------

// softmax of policy.rs:10-19 over `n` values already staged in `buf` (shared memory):
// max, exp(x - max) with the libm-exact expf, SEQUENTIAL f32 sum, division.
__device__ __forceinline__ bool warp_softmax_inplace(float* buf, int n, int lane) {
    float mx = -__int_as_float(0x7f800000);
    bool bad = false;
    for (int i = lane; i < n; i += 32) {
        const float x = buf[i];
        bad = bad || x != x;
        mx = fmaxf(mx, x);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(FULL_MASK, mx, o));
    if (n == 0) mx = 0.0f;
    __syncwarp();
    for (int i = lane; i < n; i += 32) buf[i] = expf_libm(fsub(buf[i], mx));
    __syncwarp();
    float sum = 0.0f;
    if (lane == 0)
        for (int i = 0; i < n; i++) sum = fadd(sum, buf[i]);
    sum = __shfl_sync(FULL_MASK, sum, 0);
    for (int i = lane; i < n; i += 32) buf[i] = fdiv(buf[i], sum);
    __syncwarp();
    return !__any_sync(FULL_MASK, bad);
}

// backward_network_eval (mcts.rs:171-225) of evaluation-queue entry q of game g, in three parts so that the single-tree
// path can run the parts of different leaves at the same time (k_tree_backward); the batched search runs them back to
// back (warp_expand).
struct LeafOutputs {
    float value, variance;
    bool priors_ok;
};

// part 1, private to the entry: the heads' last step, softmax over the legal logits into `p`, outputs made finite
__device__ __forceinline__ LeafOutputs expand_outputs(const TzDev& d, int q, float* p, int lane) {
    const int n = d.n_actions[q];
    const float* lg = d.logits + (size_t)q * d.M;
    for (int i = lane; i < n; i += 32) p[i] = lg[i];
    __syncwarp();
    LeafOutputs o;
    if (d.nn_head_feat != nullptr)  // device network: the heads' last step happens here (encode.cuh)
        enc::warp_heads(d.nn_head_feat, d.nn_head_misc, d.nn_novelty_set, d.nn_novelty_idx, d.nn_rnd_unc, q, d.nn, lane, &o.value,
                        &o.variance);
    else {
        o.value = d.value[q];
        o.variance = d.variance[q];
    }
    // NaN / infinite network outputs: the reference panics (net6_simhash.rs:304, NotNan).  Here the error bit is
    // raised and the outputs are replaced by finite ones (uniform priors, zero logits / value / variance), so that no
    // NaN ever enters a tree: comparisons against NaN would derail the argmax / ranking code that indexes the arena.
    o.priors_ok = warp_softmax_inplace(p, n, lane);
    {
        bool finite = true;
        for (int i = lane; i < n; i += 32) finite = finite && p[i] >= 0.0f && p[i] <= 1.0f;  // false for NaN
        o.priors_ok = o.priors_ok && __all_sync(FULL_MASK, finite);
    }
    const bool value_ok = fabsf(o.value) <= 3.0e38f && o.variance >= 0.0f && o.variance <= 3.0e38f;  // false for NaN
    if (!o.priors_ok || !value_ok) {
        flag_error(d, TZ_ERR_NAN, lane);
        if (!o.priors_ok) {
            const float uniform = fdiv(1.0f, (float)(n > 0 ? n : 1));
            for (int i = lane; i < n; i += 32) p[i] = uniform;
            __syncwarp();
        }
        if (!value_ok) {
            o.value = 0.0f;
            o.variance = 0.0f;
        }
    }
    return o;
}

// part 2, the leaf (mcts.rs:190-217, node/mod.rs:66-79): running mean / std of the leaf, its children created in the
// arena.  In two halves for the single-tree wavefront: (a) reads the leaf and writes only fresh arena slots, (b) stores
// the leaf's own words.  False when the arena is full (reported; nothing is backed up then).
struct LeafUpdate {
    float mean, std_dev;
    uint32_t start;
};

__device__ __forceinline__ bool expand_leaf_children(const TzDev& d, int g, int q, uint32_t leaf, const float* p,
                                                     const LeafOutputs& o, int lane, LeafUpdate* u) {
    const int n = d.n_actions[q];
    const GameTree t = game_tree(d.arena, g);
    const float* lg = d.logits + (size_t)q * d.M;
    const uint16_t* act = d.actions + (size_t)q * d.M;
    // the leaf's evaluation is a Value here
    const float nv = (float)t.visits[leaf];
    float m = __uint_as_float(t.eval[leaf]);
    float sd = t.std_dev[leaf];
    m = fadd(m, fdiv(fadd(fneg(m), o.value), nv));
    sd = fadd(sd, fdiv(fadd(fneg(sd), fsqrt(o.variance)), nv));
    uint32_t start = 0;
    if (lane == 0) {
        start = d.arena.next_slot[g];
        if (start + (uint32_t)n > d.arena.cap) {
            start = 0;
        } else {
            d.arena.next_slot[g] = start + (uint32_t)n;
            d.counters[(size_t)g * 4 + 3] += 1;
        }
    }
    start = __shfl_sync(FULL_MASK, start, 0);
    if (start == 0) {
        flag_error(d, TZ_ERR_ARENA_FULL, lane);
        return false;
    }
    const uint32_t child_eval = __float_as_uint(fneg(m));
    for (int i = lane; i < n; i += 32) {
        const uint32_t c = start + i;
        t.eval[c] = child_eval;
        t.meta[c] = tz_meta(act[i], TZ_E_VALUE, 0);
        t.visits[c] = 0;
        t.prob[c] = p[i];
        t.std_dev[c] = sd;
        t.logit[c] = o.priors_ok ? lg[i] : 0.0f;
        t.first[c] = 0;
    }
    u->mean = m;
    u->std_dev = sd;
    u->start = start;
    return true;
}

__device__ __forceinline__ void expand_leaf_store(const TzDev& d, int g, int q, uint32_t leaf, const LeafUpdate& u, int lane) {
    const GameTree t = game_tree(d.arena, g);
    if (lane == 0) {
        t.eval[leaf] = __float_as_uint(u.mean);
        t.std_dev[leaf] = u.std_dev;
        t.meta[leaf] = tz_meta(tz_meta_move(t.meta[leaf]), TZ_E_VALUE, (uint32_t)d.n_actions[q]);
        t.first[leaf] = u.start;
    }
    __syncwarp();
}

__device__ __forceinline__ bool expand_leaf(const TzDev& d, int g, int q, uint32_t leaf, const float* p,
                                            const LeafOutputs& o, int lane) {
    LeafUpdate u;
    if (!expand_leaf_children(d, g, q, leaf, p, o, lane, &u)) return false;
    expand_leaf_store(d, g, q, leaf, u, lane);
    return true;
}

// part 3 starts from this: what the leaf hands to its parent (mcts.rs:219-224)
__device__ __forceinline__ Propagated expand_propagated(const LeafOutputs& o) {
    Propagated pr;
    pr.eval = ev_value(fmul(o.value, 0.997f));
    pr.variance = fmul(fmul(o.variance, 0.997f), 0.997f);
    return pr;
}

__device__ __forceinline__ void warp_expand(const TzDev& d, int g, int q, const uint32_t* traj, int len, float* p,
                                            int lane) {
    const LeafOutputs o = expand_outputs(d, q, p, lane);
    if (!expand_leaf(d, g, q, traj[len - 1], p, o, lane)) return;
    warp_backup(game_tree(d.arena, g), traj, len, expand_propagated(o), lane);
}

__global__ void __launch_bounds__(32 * WPB) k_expand(TzDev d) {
    __shared__ float s_p[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WPB + warp;
    if (q >= *d.nn_count) return;
    const int g = d.nn_queue[q];
    warp_expand(d, g, q, d.traj + (size_t)g * TZ_MAX_DEPTH, d.traj_len[g], s_p[warp], lane);
}

// ---- search trees: Node::simulate_simple / simulate_batch (mcts.rs:235-328), one CTA per tree ------------------

// Up to `max_forwards` descents of ONE tree with the reference's SEQUENTIAL semantics: the visit increments of earlier
// descents steer later ones (its only "virtual loss"), known results are backed up at once, up to batch_size leaves
// need the network.  CTA t searches the tree of game d.tree_game[t]; the trees of one launch share nothing but the
// evaluation queue.  Each leaf takes a queue slot q of its own (atomicAdd on nn_count, after its commit, so the queue
// is dense over all trees in some order), its path goes to traj[q], and d.tree_slot[t * batch_size + i] = q records
// the tree's i-th leaf in commit order, d.tree_fill[t] how many there are: k_tree_backward walks them in that order.
// Which slot a leaf lands in does not change its network outputs (DESIGN §5), so neither does the order across trees.
//
// One warp doing them one after the other is bound by the latency of its own dependent loads (~12 us per descent), so
// TREE_WARPS warps of one CTA run consecutive descents as a wavefront, speculatively, and commit them in order:
//   * a descent is a chain inc_0, look_0, inc_1, look_1, ...: inc_k counts its visit of the path's node at level k,
//     look_k reads that node and its children (level k+1) and picks one.  Descent i runs inc_0 after every earlier
//     descent's inc_0 and look_k after every earlier descent's inc_(k+1) or end (tree_earlier_reached): then look_k sees
//     the level-(k+1) increments of every earlier descent and of no later one (descent i+1's inc_(k+1) follows ITS
//     look_k, which follows this descent's inc_(k+1)), and the count inc_k returns -- used by look_k instead of a second
//     read -- holds exactly the earlier descents' visits.  Without known results this is the sequential order of every
//     read and write, with consecutive descents one look apart.
//   * a descent is final only when it COMMITS, in index order.  A leaf that needs the network commits by taking the
//     next queue slot (its move list was generated while it waited).  A known result commits by (1) voiding every
//     later descent in flight -- they saw evaluations its backup is about to change -- which take back their visit
//     increments (and a terminal evaluation they may have stored on the way), (2) backing up, (3) letting them start
//     again.  The batch being full, the forward budget being used up, or a committed error void the rest for good.
// Control words in shared memory (volatile):
//   fprog[w]  descent that warp w runs: index * 1024 + increments done (1000 = over)
//   commit    index of the next descent to commit          filled   queue entries taken
//   gen       bumped by every voiding                      resume   last generation whose voiding is complete
//   acks      warps that have taken back their descent since the last voiding          stop   no more descents
#ifndef TREE_WARPS
#define TREE_WARPS 8
#endif
#define TREE_SPIN_LIMIT (1 << 24)

struct TreeCtl {
    int nw;  // warps of this launch (<= TREE_WARPS; fewer only in tests, to vary the interleaving)
    volatile int* fprog;
    volatile int* commit;
    volatile int* filled;
    volatile int* gen;
    volatile int* resume;
    volatile int* acks;
    volatile int* stop;
};

enum { TREE_NEEDS = 0, TREE_KNOWN = 1, TREE_ERROR = -1, TREE_VOID = -2 };

// lane 0 spins until `cond` holds; false when this descent has been voided meanwhile (or the wait gave up)
template <typename Cond>
__device__ __forceinline__ bool tree_spin(const TzDev& d, const TreeCtl& c, int my_gen, int lane, Cond cond) {
    int ok = 1;
    if (lane == 0) {
        int spins = 0;
        while (true) {
            if (*c.gen != my_gen) {
                ok = 0;
                break;
            }
            if (cond()) break;
            if (++spins > TREE_SPIN_LIMIT) {  // never seen; ends the whole launch instead of hanging the GPU
                atomicOr(d.status, TZ_ERR_NETWORK_STALL);
                *c.stop = 1;
                ok = 0;
                break;
            }
        }
    }
    ok = __shfl_sync(FULL_MASK, ok, 0);
    __threadfence_block();
    return ok != 0;
}

// Have all descents before `it` made at least `need` increments, or ended?  The nearest one still going decides: its
// own looks waited for the ones before it.  (One that has ENDED says nothing about the ones before it -- its path may
// just be shorter than theirs -- so the scan goes on behind it; descents a whole round of warps back have committed.)
__device__ __forceinline__ bool tree_earlier_reached(const TreeCtl& c, int it, int need) {
    for (int j = it - 1; j >= 0 && j > it - c.nw; j--) {
        const int v = c.fprog[j % c.nw];
        if (v >= j * 1024 + 1000) continue;
        return v >= j * 1024 + need;
    }
    return true;
}

__device__ __forceinline__ void tree_fpublish(const TreeCtl& c, int it, int steps, int lane) {
    __threadfence_block();
    __syncwarp();
    if (lane == 0) c.fprog[it % c.nw] = it * 1024 + steps;
}

// Node::forward (mcts.rs:107-138) as warp_forward does it, as a chain inc_0, look_0, inc_1, look_1, ...: inc_k counts
// the visit of the path's node at level k (and keeps the new count for look_k's exploration term), look_k reads that
// node and its children and picks the next one.  `undo_*`: the terminal evaluation this descent stored on an
// uninitialised node, to be taken back if the descent is voided.
__device__ __forceinline__ int tree_descend(const TzDev& d, const GameTree& t, const TreeCtl& c, TzState* st, uint32_t* traj,
                                            int it, int my_gen, float beta, int lane, int* out_len, Ev* known_ev,
                                            uint32_t* err_bit, uint32_t* undo_slot, uint32_t* undo_words) {
    int len = 0;
    uint32_t slot = 0;
    *undo_slot = 0xffffffffu;
    *out_len = 0;
    while (true) {
        // inc_len: after the previous descent's own inc_len (for level 0; deeper ones follow from the look rule)
        if (len >= TZ_MAX_DEPTH) {
            *err_bit = TZ_ERR_DEPTH;
            return TREE_ERROR;
        }
        if (it > 0 && len == 0) {
            if (!tree_spin(d, c, my_gen, lane, [=]() { return tree_earlier_reached(c, it, 1); })) return TREE_VOID;
        }
        // the node's own words ride along with the increment: nothing but a known result's commit changes them during
        // this launch, and that voids this descent anyway
        const uint32_t meta = t.meta[slot];
        const uint32_t eval_bits = t.eval[slot];
        uint32_t pv = 0;
        if (lane == 0) {
            // atomic: a voided descent may be taking its increment of this very node (the root, say) back right now
            pv = atomicAdd(&t.visits[slot], 1u) + 1u;
            traj[len] = slot;
        }
        len++;
        *out_len = len;
        // the move that leads here is played while the increment is on its way (the next descent waits for the
        // increment, not for the board)
        const bool applied = len == 1 || warp_apply(st, d.n, (uint16_t)tz_meta_move(meta), lane);
        pv = __shfl_sync(FULL_MASK, pv, 0);
        tree_fpublish(c, it, len, lane);
        if (!applied) {
            *err_bit = TZ_ERR_BAD_MOVE;
            return TREE_ERROR;
        }
        // look_(len-1): after every earlier descent's inc_len, or its end
        if (it > 0) {
            const int need = len + 1;
            if (!tree_spin(d, c, my_gen, lane, [=]() { return tree_earlier_reached(c, it, need); })) return TREE_VOID;
        }
        const uint32_t tag = tz_meta_tag(meta);
        if (tag != TZ_E_VALUE && eval_bits == 0) {  // is_terminal
            *known_ev = ev_make(tag, 0);
            return TREE_KNOWN;
        }
        if (tz_meta_nchild(meta) == 0 && tag == TZ_E_VALUE) {  // needs_initialization
            const int term = warp_terminal(st, d.n, d.half_komi, d.rev_limit, lane);
            if (term != TZ_T_NONE) {
                *known_ev = ev_make(term == TZ_T_WIN ? TZ_E_WIN : (term == TZ_T_LOSS ? TZ_E_LOSS : TZ_E_DRAW), 0);
                undo_words[0] = t.eval[slot];
                undo_words[1] = t.meta[slot];
                undo_words[2] = __float_as_uint(t.std_dev[slot]);
                *undo_slot = slot;
                if (lane == 0) {
                    node_set_eval(t, slot, *known_ev);
                    t.std_dev[slot] = 0.0f;
                }
                __syncwarp();
                return TREE_KNOWN;
            }
            return TREE_NEEDS;
        }
        bool nan_seen;
        const int idx = warp_select_puct(t, slot, beta, d.ln_table, lane, &nan_seen, (long long)pv);
        if (nan_seen) flag_error(d, TZ_ERR_NAN, lane);
        if (idx < 0) {
            *err_bit = TZ_ERR_NO_CHILD;
            return TREE_ERROR;
        }
        slot = t.first[slot] + (uint32_t)idx;
    }
}

// a voided descent takes back what it did to the tree (other voided descents do the same at the same time, and they
// all went through the root: atomics)
__device__ __forceinline__ void tree_take_back(const GameTree& t, const uint32_t* traj, int len, uint32_t undo_slot,
                                               const uint32_t* undo_words, int lane) {
    for (int i = lane; i < len; i += 32) atomicSub(&t.visits[traj[i]], 1u);
    if (undo_slot != 0xffffffffu && lane == 0) {
        t.eval[undo_slot] = undo_words[0];
        t.meta[undo_slot] = undo_words[1];
        t.std_dev[undo_slot] = __uint_as_float(undo_words[2]);
    }
    __syncwarp();
}

struct TreeForwardSmem {
    TzState state[TREE_WARPS];
    uint16_t moves[TREE_WARPS][TZ_MAX_MOVES];
    uint32_t ranges[TREE_WARPS][TZ_MAX_SQ];
    uint32_t traj[TREE_WARPS][TZ_MAX_DEPTH];
    int fprog[TREE_WARPS];
    int ctl[6];
};

__global__ void __launch_bounds__(32 * TREE_WARPS) k_tree_forward(TzDev d, float beta, int batch_size, int max_forwards) {
    const int tree = blockIdx.x, g = d.tree_game[tree];
    extern __shared__ __align__(128) unsigned char tree_smem[];
    TreeForwardSmem& sm = *reinterpret_cast<TreeForwardSmem*>(tree_smem);
    TzState* s_state = sm.state;
    uint16_t(*s_moves)[TZ_MAX_MOVES] = sm.moves;
    uint32_t(*s_ranges)[TZ_MAX_SQ] = sm.ranges;
    uint32_t(*s_traj)[TZ_MAX_DEPTH] = sm.traj;
    int* s_fprog = sm.fprog;
    int* s_ctl = sm.ctl;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    TreeCtl c;
    c.nw = blockDim.x >> 5;
    c.fprog = s_fprog;
    c.commit = s_ctl + 0;
    c.filled = s_ctl + 1;
    c.gen = s_ctl + 2;
    c.resume = s_ctl + 3;
    c.acks = s_ctl + 4;
    c.stop = s_ctl + 5;
    if (threadIdx.x < 6) s_ctl[threadIdx.x] = 0;
    if (lane == 0) s_fprog[warp] = -1;
    if (threadIdx.x == 0) d.tree_fill[tree] = 0;  // the committing warp that ends the batch writes the real count
    __syncthreads();
    const GameTree t = game_tree(d.arena, g);
    unsigned long long* ctr = d.counters + (size_t)g * 4;  // only the committing warp touches the tree's counters
    TzState* st = &s_state[warp];
    uint32_t* traj = s_traj[warp];
    if (max_forwards <= 0 || batch_size <= 0) return;

    int it = warp;
    int acked_gen = 0;  // lane 0: the last voiding this warp has acknowledged (every warp acknowledges every one)
    while (true) {
        // (re)start: not while a voiding is under way; a warp with nothing left keeps answering until the end
        int my_gen = 0, stopped = 0;
        if (lane == 0) {
            int spins = 0;
            while (true) {
                stopped = *c.stop;
                my_gen = *c.gen;
                if (stopped) break;
                if (*c.resume != my_gen) {  // a voiding is under way and this warp holds nothing to take back
                    if (acked_gen != my_gen) {
                        acked_gen = my_gen;
                        atomicAdd((int*)c.acks, 1);
                    }
                } else if (it < max_forwards) {
                    break;
                } else {
                    __nanosleep(200);
                }
                if (++spins > TREE_SPIN_LIMIT) {
                    atomicOr(d.status, TZ_ERR_NETWORK_STALL);
                    *c.stop = 1;
                    stopped = 1;
                    break;
                }
            }
        }
        my_gen = __shfl_sync(FULL_MASK, my_gen, 0);
        stopped = __shfl_sync(FULL_MASK, stopped, 0);
        __threadfence_block();
        if (stopped) return;
        tree_fpublish(c, it, 0, lane);
        warp_load_state(st, &d.env[g], lane);
        int len = 0;
        Ev known_ev = ev_value(0.0f);
        uint32_t err_bit = 0, undo_slot = 0xffffffffu, undo_words[3] = {0, 0, 0};
        int res = tree_descend(d, t, c, st, traj, it, my_gen, beta, lane, &len, &known_ev, &err_bit, &undo_slot, undo_words);
        int cnt = 0;
        if (res != TREE_VOID) {
            tree_fpublish(c, it, 1000, lane);
            if (res == TREE_NEEDS) {
                // Forward::NeedsNetwork: the move list and what the input encoding needs, while waiting for the turn
                cnt = warp_movegen(st, d.n, s_moves[warp], lane, s_ranges[warp]);
                if (cnt >= 0 && cnt <= d.M) {
                    const TzBoards b = warp_boards(st, d.nn, lane);
                    if (lane == 0)
                        enc::store_position_scalars(st, __popcll(b.flat[0]) - __popcll(b.flat[1]), d.n, d.half_komi, d.nn_f16);
                    __syncwarp();
                }
            }
            volatile int* commit = c.commit;
            if (!tree_spin(d, c, my_gen, lane, [=]() { return *commit == it; })) res = TREE_VOID;
        }
        if (res == TREE_VOID) {
            tree_take_back(t, traj, len, undo_slot, undo_words, lane);
            tree_fpublish(c, it, 0, lane);
            if (lane == 0 && acked_gen != my_gen + 1) {
                acked_gen = my_gen + 1;  // one voiding at a time: the next one cannot start before this one is complete
                atomicAdd((int*)c.acks, 1);
            }
            __syncwarp();
            continue;  // the same descent again, once the voiding is complete (or never, when stopped)
        }

        // ---- commit: this descent is the oldest one in flight, everything before it is final ----
        bool stop = false;
        int filled = *c.filled;
        const int q = filled;
        if (lane == 0) ctr[0] += 1;
        if (res == TREE_ERROR) {
            flag_error(d, err_bit, lane);
            stop = true;
        } else if (res == TREE_KNOWN) {
            // void the later descents, wait until they have taken their increments back, then back up
            if (lane == 0) {
                *c.acks = 0;
                __threadfence_block();
                *c.gen = my_gen + 1;
                int spins = 0;
                while (*c.acks < c.nw - 1 && ++spins <= TREE_SPIN_LIMIT) {
                }
                if (spins > TREE_SPIN_LIMIT) atomicOr(d.status, TZ_ERR_NETWORK_STALL);
                ctr[2] += 1;
            }
            __syncwarp();
            __threadfence_block();
            Propagated p;
            p.eval = known_ev;
            p.variance = 0.0f;
            warp_backup(t, traj, len, p, lane);
        } else {
            if (lane == 0) ctr[1] += 1;
            if (cnt < 0 || cnt > d.M) {
                flag_error(d, TZ_ERR_TOO_MANY_MOVES, lane);
                stop = true;
            } else {
                filled = q + 1;
            }
        }
        stop = stop || filled >= batch_size || it + 1 >= max_forwards;
        __threadfence_block();
        __syncwarp();
        if (lane == 0) {
            *c.filled = filled;
            if (stop) {
                d.tree_fill[tree] = filled;
                *c.stop = 1;
                __threadfence_block();
                if (res != TREE_KNOWN) *c.gen = my_gen + 1;  // whoever is still descending gives up and takes it back
            } else {
                *c.commit = it + 1;
                __threadfence_block();
                if (res == TREE_KNOWN) *c.resume = my_gen + 1;
            }
        }
        __syncwarp();
        if (res == TREE_NEEDS && filled > q) {
            // the tree's entry q is this descent's alone from here on: taking a queue slot and filling it keeps nobody
            // waiting.  (A leaf with too many moves is reported, never truncated, and gets no entry: it ended the batch.)
            int slot = 0;
            if (lane == 0) {
                slot = atomicAdd(d.nn_count, 1);
                d.tree_slot[(size_t)tree * batch_size + q] = slot;
                d.nn_queue[slot] = g;
                d.n_actions[slot] = cnt;
                d.traj_len[slot] = len;
            }
            slot = __shfl_sync(FULL_MASK, slot, 0);
            for (int sq = lane; sq < TZ_MAX_SQ; sq += 32) d.sq_ranges[(size_t)slot * TZ_MAX_SQ + sq] = s_ranges[warp][sq];
            warp_store_state(&d.leaf_state[slot], st, lane);
            uint16_t* out = d.actions + (size_t)slot * d.M;
            for (int i = lane; i < cnt; i += 32) out[i] = s_moves[warp][i];
            uint32_t* tq = d.traj + (size_t)slot * TZ_MAX_DEPTH;
            for (int i = lane; i < len; i += 32) tq[i] = traj[i];
            __syncwarp();
        }
        if (stop) return;
        it += c.nw;
    }
}

// backward_network_eval of one tree's queued leaves IN ITS COMMIT ORDER (they share the tree: every running mean and
// every solver scan sees what the earlier leaves of the batch left), by TREE_WARPS warps of the tree's CTA as a wavefront
// (entry q below is the tree's q-th leaf, at queue slot d.tree_slot[t * batch_size + q]):
//   * the heads, the softmax and the sanitising of an entry touch nothing shared and run at once for TREE_WARPS entries;
//   * entry q works on depth e of its path (leaf step at e = len-1, then the parents up to the root at 0) in two halves:
//     it READS the node at depth e and its children at depth e+1 once entry q-1 has finished depth e (by induction so
//     have all earlier entries: what they wrote on both levels is final and visible -- fence + progress word in shared
//     memory), and it STORES the node at depth e once entry q-1 has finished depth e-1, because until then that entry's
//     solver scan at depth e-1 may still be reading this node as one of its children.  So consecutive entries run one
//     step apart, the reads and the arithmetic of one overlapping the step above it of the other.  The arena allocations
//     happen in the leaf steps, hence in order; fresh child slots are written in the read half (nobody can reach them).
// progress word of the warp that owns entry q: q * 1024 + (1000 - last finished depth), monotonic over its entries.
__device__ __forceinline__ int tree_progress(int q, int finished_depth) { return q * 1024 + (1000 - finished_depth); }

// wait until entry `q - 1` has finished depth `need` (-1 = all of it); false when the wait gave up
__device__ __forceinline__ bool tree_wait_pred(const TzDev& d, volatile int* prog, int nw, int q, int need, int lane) {
    bool ok = true;
    if (q > 0) {
        if (lane == 0) {
            const int want = tree_progress(q - 1, need);
            int spins = 0;
            while (prog[(q - 1) % nw] < want)
                if (++spins > TREE_SPIN_LIMIT) {
                    ok = false;
                    break;
                }
        }
        ok = __shfl_sync(FULL_MASK, ok ? 1 : 0, 0) != 0;
        if (!ok) flag_error(d, TZ_ERR_NETWORK_STALL, lane);
    }
    __threadfence_block();
    return ok;
}

__device__ __forceinline__ void tree_publish(volatile int* prog, int nw, int q, int finished_depth, int lane) {
    __threadfence_block();
    __syncwarp();
    if (lane == 0) prog[q % nw] = tree_progress(q, finished_depth);
}

struct TreeBackwardSmem {
    float p[TREE_WARPS][TZ_MAX_MOVES];
    int prog[TREE_WARPS];
};

__global__ void __launch_bounds__(32 * TREE_WARPS) k_tree_backward(TzDev d, int batch_size) {
    extern __shared__ __align__(128) unsigned char tree_smem[];
    TreeBackwardSmem& sm = *reinterpret_cast<TreeBackwardSmem*>(tree_smem);
    float(*s_p)[TZ_MAX_MOVES] = sm.p;
    int* s_prog = sm.prog;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tree = blockIdx.x, g = d.tree_game[tree];
    const int count = d.tree_fill[tree];
    const int* slots = d.tree_slot + (size_t)tree * batch_size;
    volatile int* prog = s_prog;
    if (lane == 0) s_prog[warp] = -1;
    __syncthreads();
    const GameTree t = game_tree(d.arena, g);
    const int nw = blockDim.x >> 5;
    for (int q = warp; q < count; q += nw) {
        const int slot = slots[q];
        const uint32_t* traj = d.traj + (size_t)slot * TZ_MAX_DEPTH;
        const int len = d.traj_len[slot];
        const LeafOutputs o = expand_outputs(d, slot, s_p[warp], lane);
        const uint32_t leaf = traj[len - 1];
        LeafUpdate u;
        bool ok = tree_wait_pred(d, prog, nw, q, len - 1, lane);  // reads at the leaf's depth
        ok = ok && expand_leaf_children(d, g, slot, leaf, s_p[warp], o, lane, &u);
        ok = tree_wait_pred(d, prog, nw, q, len - 2, lane) && ok;  // stores at the leaf's depth
        if (ok) expand_leaf_store(d, g, slot, leaf, u, lane);
        Propagated pr = expand_propagated(o);
        for (int e = len - 2; ok && e >= 0; e--) {
            tree_publish(prog, nw, q, e + 1, lane);
            PendingNode w;
            ok = tree_wait_pred(d, prog, nw, q, e, lane);  // reads at depth e (and e+1)
            if (ok) pr = warp_propagate_compute(t, traj[e], pr, lane, &w);
            ok = ok && tree_wait_pred(d, prog, nw, q, e - 1, lane);  // stores at depth e
            if (ok) warp_propagate_store(t, w, lane);
        }
        tree_publish(prog, nw, q, -1, lane);  // also after an error: nobody waits for ever
    }
}

// ---- Gumbel top-k and sequential halving -----------------------------------------------

__device__ __forceinline__ uint64_t rng_hash(uint64_t seed, uint64_t a, uint64_t b, uint64_t c) {
    uint64_t h = tz_mix64(seed ^ 0x9e3779b97f4a7c15ULL);
    h = tz_mix64(h ^ (a * 0xbf58476d1ce4e5b9ULL));
    h = tz_mix64(h ^ (b * 0x94d049bb133111ebULL));
    return tz_mix64(h ^ (c * 0xd6e8feb86659fd93ULL));
}

// Gumbel(0,1) noise for every (game, child index): the reference draws from `rand`
// (batched.rs:226-227), whose stream is not pinned, so this is our own counter-based
// generator keyed by the GLOBAL game id (sharded == unsharded).
__global__ void k_gumbel_noise(TzDev d, float* out, int stride, unsigned long long seed,
                               unsigned long long counter) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)d.G * stride) return;
    const int g = (int)(idx / stride), i = (int)(idx % stride);
    const uint64_t h = rng_hash(seed, (uint64_t)(d.game_base + g), counter, (uint64_t)i);
    const float u = ((float)(h >> 40) + 0.5f) * (1.0f / 16777216.0f);  // (0,1)
    out[idx] = -logf(-logf(u));
}

// stable descending rank of element `i` among `n` keys in shared memory
__device__ __forceinline__ int stable_desc_rank(const float* keys, int n, int i) {
    const float k = keys[i];
    int rank = 0;
    for (int j = 0; j < n; j++) {
        const float o = keys[j];
        rank += (o > k) || (o == k && j < i);
    }
    return rank;
}

__global__ void __launch_bounds__(32 * WPB) k_gumbel_init(TzDev d, int k, const float* gumbel, int stride) {
    __shared__ float s_key[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    const GameTree t = game_tree(d.arena, g);
    const int n = (int)tz_meta_nchild(t.meta[0]);
    const uint32_t first = t.first[0];
    float* keys = s_key[warp];
    bool bad = false;
    // batched.rs:233-239 zips one draw with every child: a caller whose rows are shorter than a root's child list has
    // not supplied them -- reported (never another game's noise), the children without a draw are ordered last
    if (n > stride) flag_error(d, TZ_ERR_TOO_MANY_MOVES, lane);
    for (int i = lane; i < n; i += 32) {
        const float key = i < stride ? fadd(t.logit[first + i], gumbel[(size_t)g * stride + i]) : -__int_as_float(0x7f800000);
        bad = bad || key != key;
        // a NaN key (NaN noise, or -inf logit + inf noise) would give several children the same rank and leave
        // slots of the candidate set unwritten: order it last instead (the error bit is raised below)
        keys[i] = key != key ? -__int_as_float(0x7f800000) : key;
    }
    if (__any_sync(FULL_MASK, bad)) flag_error(d, TZ_ERR_NAN, lane);
    __syncwarp();
    for (int i = lane; i < n; i += 32) {
        const int r = stable_desc_rank(keys, n, i);
        if (r < k) {
            d.set_child[(size_t)g * TZ_MAX_K + r] = (uint16_t)i;
            d.set_key[(size_t)g * TZ_MAX_K + r] = keys[i];
        }
    }
    if (lane == 0) d.set_len[g] = n < k ? n : k;
}

__global__ void __launch_bounds__(32 * WPB) k_halve(TzDev d, const float* betas, float visits, int remaining) {
    __shared__ float s_key[WPB][TZ_MAX_K];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    const GameTree t = game_tree(d.arena, g);
    const uint32_t first = t.first[0];
    const int len = d.set_len[g];
    const float beta = betas ? betas[g] : 0.0f;
    float* keys = s_key[warp];
    uint16_t child[TZ_MAX_K / 32];
    float base[TZ_MAX_K / 32];
#pragma unroll
    for (int r = 0; r < TZ_MAX_K / 32; r++) {
        const int j = lane + 32 * r;
        if (j < len) {
            child[r] = d.set_child[(size_t)g * TZ_MAX_K + j];
            base[r] = d.set_key[(size_t)g * TZ_MAX_K + j];
            const uint32_t c = first + child[r];
            const float q = ev_notnan(ev_negate(node_eval(t, c)));
            // sigma_select (policy.rs:121-128)
            const float sig = fmul(fadd(q, fmul(t.std_dev[c], beta)), fadd(50.0f, visits));
            const float key = fadd(base[r], sig);
            if (key != key) flag_error(d, TZ_ERR_NAN, 0);  // e.g. a NaN beta from the host
            keys[j] = key != key ? -__int_as_float(0x7f800000) : key;
        }
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < TZ_MAX_K / 32; r++) {
        const int j = lane + 32 * r;
        if (j < len) {
            const int rank = stable_desc_rank(keys, len, j);
            if (rank < remaining) {
                d.set_child[(size_t)g * TZ_MAX_K + rank] = child[r];
                d.set_key[(size_t)g * TZ_MAX_K + rank] = base[r];
            }
        }
    }
    if (lane == 0) d.set_len[g] = len < remaining ? len : remaining;
}

// root statistics recompute of batched.rs:373-406; warp-convergent
__device__ __forceinline__ void warp_root_recompute(const TzDev& d, const GameTree& t, float* buf, int lane) {
    const uint32_t meta = t.meta[0];
    const int n = (int)tz_meta_nchild(meta);
    const uint32_t first = t.first[0];
    uint32_t sum = 0;
    for (int i = lane; i < n; i += 32) sum += t.visits[first + i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(FULL_MASK, sum, o);
    const int flags = warp_children_flags(t, first, n, lane);
    if (lane == 0) t.visits[0] = sum + 1;
    if (n == 0) return;  // reference: `.min().unwrap()` panics; callers flag the empty root
    if ((flags & 2) || (flags & 1)) {
        Ev m;
        warp_min_child(t, first, n, lane, &m);
        if (lane == 0) {
            node_set_eval(t, 0, ev_negate(m));
            t.std_dev[0] = 0.0f;
        }
    } else {
        // sum of p, then sum of p*q, each SEQUENTIALLY over the visited children
        const float skip = __int_as_float(0x7fc00000);  // NaN marks an unvisited child
        for (int i = lane; i < n; i += 32) buf[i] = t.visits[first + i] > 0 ? t.prob[first + i] : skip;
        __syncwarp();
        float sum_p = 0.0f;
        if (lane == 0)
            for (int i = 0; i < n; i++) {
                const float x = buf[i];
                if (x == x) sum_p = fadd(sum_p, x);
            }
        __syncwarp();
        for (int i = lane; i < n; i += 32)
            if (t.visits[first + i] > 0)
                buf[i] = fmul(t.prob[first + i], ev_to_f32(ev_negate(node_eval(t, first + i))));
        __syncwarp();
        if (lane == 0) {
            float wq = 0.0f;
            for (int i = 0; i < n; i++) {
                const float x = buf[i];
                if (x == x) wq = fadd(wq, x);
            }
            node_set_eval(t, 0, ev_value(fdiv(wq, sum_p)));
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(32 * WPB) k_finalize(TzDev d, uint16_t* out_moves) {
    __shared__ float s_buf[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    const GameTree t = game_tree(d.arena, g);
    if (d.set_len[g] != 1) {
        flag_error(d, TZ_ERR_SET_EMPTY, lane);
        if (lane == 0) out_moves[g] = 0xffff;
    } else if (lane == 0) {
        const uint32_t c = t.first[0] + d.set_child[(size_t)g * TZ_MAX_K];
        out_moves[g] = (uint16_t)tz_meta_move(t.meta[c]);
    }
    warp_root_recompute(d, t, s_buf[warp], lane);
}

// ---- step: re-root with subtree reuse ---------------------------------------------------

__device__ __forceinline__ void copy_node(const GameTree& dst, uint32_t to, const GameTree& src, uint32_t from) {
    dst.eval[to] = src.eval[from];
    dst.meta[to] = src.meta[from];
    dst.visits[to] = src.visits[from];
    dst.prob[to] = src.prob[from];
    dst.std_dev[to] = src.std_dev[from];
    dst.logit[to] = src.logit[from];
    dst.first[to] = src.first[from];
}

// `Game::play` of a move that came from the host: legal iff it is one of `possible_moves` (warp_apply itself
// trusts its move, as the search only ever applies generated ones).  Leaves the position untouched when illegal.
__device__ __forceinline__ bool warp_apply_checked(TzState* st, int n, uint16_t mv, uint16_t* scratch, int lane) {
    const int cnt = warp_movegen(st, n, scratch, lane);
    __syncwarp();
    bool found = false;
    for (int i = lane; i < cnt; i += 32) found = found || scratch[i] == mv;
    if (!__any_sync(FULL_MASK, found)) return false;
    return warp_apply(st, n, mv, lane);
}

__global__ void __launch_bounds__(32 * WPB) k_step(TzDev d, const uint16_t* moves, const uint8_t* mask) {
    __shared__ TzState s_state[WPB];
    __shared__ uint16_t s_moves[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G || (mask && !mask[g])) return;
    const int half = d.arena.half[g];
    const GameTree src = game_tree_half(d.arena, g, half);
    const uint32_t rmeta = src.meta[0];
    if (tz_meta_tag(rmeta) != TZ_E_VALUE && src.eval[0] == 0) return;  // terminal root: batched.rs:139
    const uint16_t mv = moves[g];
    // the move comes from the host: "Action should be valid" (env.rs:44).  Checked before the tree is touched, so an
    // illegal move leaves tree and position as they were.
    TzState* st = &s_state[warp];
    warp_load_state(st, &d.env[g], lane);
    {
        const int cnt = warp_movegen(st, d.n, s_moves[warp], lane);
        __syncwarp();
        bool legal = false;
        for (int i = lane; i < cnt; i += 32) legal = legal || s_moves[warp][i] == mv;
        if (!__any_sync(FULL_MASK, legal)) {
            flag_error(d, TZ_ERR_BAD_MOVE, lane);
            return;
        }
    }
    // Node::descend (node/mod.rs:95-102)
    const int n = (int)tz_meta_nchild(rmeta);
    const uint32_t first = src.first[0];
    int found = 0x7fffffff;
    for (int i = lane; i < n; i += 32)
        if (tz_meta_move(src.meta[first + i]) == mv && i < found) found = i;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) found = min(found, __shfl_xor_sync(FULL_MASK, found, o));
    if (found == 0x7fffffff) {
        if (lane == 0) {
            node_reset(src, 0);
            d.arena.next_slot[g] = 1;
        }
    } else {
        // Cheney copy of the kept subtree into the other half, breadth first
        const GameTree dst = game_tree_half(d.arena, g, half ^ 1);
        if (lane == 0) copy_node(dst, 0, src, first + (uint32_t)found);
        __syncwarp();
        uint32_t scan = 0, alloc = 1;
        while (scan < alloc) {
            const uint32_t s = scan + lane;
            uint32_t nch = 0, oldf = 0;
            if (s < alloc) {
                nch = tz_meta_nchild(dst.meta[s]);
                oldf = dst.first[s];
            }
            uint32_t incl = nch;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(FULL_MASK, incl, o);
                if (lane >= o) incl += v;
            }
            const uint32_t total = __shfl_sync(FULL_MASK, incl, 31);
            const uint32_t newf = alloc + incl - nch;
            if (nch > 0) dst.first[s] = newf;
            uint32_t has = __ballot_sync(FULL_MASK, nch > 0);
            while (has) {
                const int L = __ffs(has) - 1;
                has &= has - 1;
                const uint32_t of = __shfl_sync(FULL_MASK, oldf, L);
                const uint32_t nf = __shfl_sync(FULL_MASK, newf, L);
                const uint32_t cnt = __shfl_sync(FULL_MASK, nch, L);
                for (uint32_t i = lane; i < cnt; i += 32) copy_node(dst, nf + i, src, of + i);
            }
            const uint32_t before = alloc;
            alloc += total;
            scan = scan + 32 < before ? scan + 32 : before;
            __syncwarp();
        }
        if (lane == 0) {
            d.arena.half[g] = (uint8_t)(half ^ 1);
            d.arena.next_slot[g] = alloc;
        }
    }
    // replay.push(action); env.step(action)
    if (!warp_apply(st, d.n, mv, lane)) flag_error(d, TZ_ERR_BAD_MOVE, lane);
    warp_store_state(&d.env[g], st, lane);
    if (lane == 0) {
        const int rl = d.replay_len[g];
        if (rl < TZ_MAX_PLIES) {
            d.replay[(size_t)g * TZ_MAX_PLIES + rl] = mv;
            d.replay_len[g] = rl + 1;
        } else {
            atomicOr(d.status, TZ_ERR_REPLAY_FULL);
        }
    }
}

// ---- positions, openings, restarts ------------------------------------------------------

__device__ __forceinline__ void state_init(TzState* s, int n) {
    // standard Tak reserves (consistent with network/repr.rs:303-409: 3 -> 10/0, 5 -> 21/1)
    const int stones = n == 3 ? 10 : n == 4 ? 15 : n == 5 ? 21 : 30;
    const int caps = n >= 5 ? 1 : 0;
    uint32_t* w = reinterpret_cast<uint32_t*>(s);
    for (int i = 0; i < (int)(sizeof(TzState) / 4); i++) w[i] = 0;
    s->stones[0] = s->stones[1] = (uint8_t)stones;
    s->caps[0] = s->caps[1] = (uint8_t)caps;
}

// env.rs:65-79: two flat placements on opposite / adjacent corners under one of 8
// symmetries (bit 0 mirror columns, bit 1 mirror rows, bit 2 transpose; the crate's own
// index order is not pinned by the reference)
__device__ __forceinline__ void warp_new_opening(TzState* st, int n, int symmetry, int adjacent, int lane) {
    if (lane == 0) state_init(st, n);
    __syncwarp();
    for (int i = 0; i < 2; i++) {
        int col = i == 0 ? 0 : (adjacent ? 0 : n - 1);
        int row = i == 0 ? 0 : n - 1;
        if (symmetry & 1) col = n - 1 - col;
        if (symmetry & 2) row = n - 1 - row;
        if (symmetry & 4) {
            const int tmp = col;
            col = row;
            row = tmp;
        }
        warp_apply(st, n, tz_mk_move(row, col, TZ_FLAT, 0), lane);
    }
}

__device__ __forceinline__ void warp_fresh_game(const TzDev& d, int g, const TzState* st, int lane) {
    warp_store_state(&d.env[g], st, lane);
    warp_store_state(&d.start_env[g], st, lane);
    if (lane == 0) {
        node_reset(game_tree(d.arena, g), 0);
        d.arena.next_slot[g] = 1;
        d.replay_len[g] = 0;
    }
}

__global__ void __launch_bounds__(32 * WPB) k_new_openings(TzDev d, const uint8_t* mask, const int* sym,
                                                           const int* adj, unsigned long long seed,
                                                           unsigned long long counter) {
    __shared__ TzState s_state[WPB];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G || (mask && !mask[g])) return;
    const uint64_t h = rng_hash(seed, (uint64_t)(d.game_base + g), counter, 0x0fe11ULL);
    warp_new_opening(&s_state[warp], d.n, sym ? sym[g] : (int)(h & 7), adj ? adj[g] : (int)((h >> 3) & 1), lane);
    warp_fresh_game(d, g, &s_state[warp], lane);
}

// Environment::new_opening_with_random_steps (env.rs:81-96) after the opening: `steps` uniformly random legal
// moves per game (stops early when a game has no legal move, i.e. is over); roots are reset.  The reference
// draws from `rand` (unpinned); here the choice is hash(seed, global game id, ply) mod the move count.
__global__ void __launch_bounds__(32 * WPB) k_random_steps(TzDev d, const uint8_t* mask, int steps,
                                                           unsigned long long seed) {
    __shared__ TzState s_state[WPB];
    __shared__ uint16_t s_moves[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G || (mask && !mask[g])) return;
    TzState* st = &s_state[warp];
    warp_load_state(st, &d.env[g], lane);
    for (int i = 0; i < steps; i++) {
        if (warp_terminal(st, d.n, d.half_komi, d.rev_limit, lane) != TZ_T_NONE) break;
        const int cnt = warp_movegen(st, d.n, s_moves[warp], lane);
        if (cnt <= 0) break;
        const uint64_t h = rng_hash(seed, (uint64_t)(d.game_base + g), (uint64_t)st->ply, 0x57e95ULL);
        warp_apply(st, d.n, s_moves[warp][h % (uint64_t)cnt], lane);
    }
    warp_fresh_game(d, g, st, lane);
}

__global__ void __launch_bounds__(32 * WPB) k_set_positions(TzDev d, const TzState* states, const uint8_t* mask) {
    __shared__ TzState s_state[WPB];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G || (mask && !mask[g])) return;
    warp_load_state(&s_state[warp], &states[g], lane);
    warp_fresh_game(d, g, &s_state[warp], lane);
}

// positions picked out of a device-resident pool (the replay buffer of `reanalyze`): game g <- pool[indices[g]], fresh root
__global__ void __launch_bounds__(32 * WPB) k_gather_positions(TzDev d, const TzState* pool, const uint32_t* indices) {
    __shared__ TzState s_state[WPB];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    warp_load_state(&s_state[warp], &pool[indices[g]], lane);
    warp_fresh_game(d, g, &s_state[warp], lane);
}

__global__ void k_reset_roots(TzDev d, const uint8_t* mask) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= d.G || (mask && !mask[g])) return;
    node_reset(game_tree(d.arena, g), 0);
    d.arena.next_slot[g] = 1;
}

// batched.rs:185-203.  A finished game's replay is parked in fin_* before the reset so the
// host can still read it; out_result (optional) receives the absolute result of the final position.
__global__ void __launch_bounds__(32 * WPB) k_restart(TzDev d, const int* sym, const int* adj,
                                                      unsigned long long seed, unsigned long long counter,
                                                      int* out_terminal, TzState* fin_start, uint16_t* fin_replay,
                                                      int* fin_len, int* out_result) {
    __shared__ TzState s_state[WPB];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    TzState* st = &s_state[warp];
    warp_load_state(st, &d.env[g], lane);
    const int term = warp_terminal(st, d.n, d.half_komi, d.rev_limit, lane);
    if (lane == 0) out_terminal[g] = term;
    if (term == TZ_T_NONE) return;
    if (out_result) {
        const int res = warp_game_result(st, d.n, d.half_komi, d.rev_limit, lane);
        if (lane == 0) out_result[g] = res;
    }
    const int rl = d.replay_len[g];
    for (int i = lane; i < rl; i += 32)
        fin_replay[(size_t)g * TZ_MAX_PLIES + i] = d.replay[(size_t)g * TZ_MAX_PLIES + i];
    if (lane == 0) fin_len[g] = rl;
    __syncwarp();
    warp_load_state(st, &d.start_env[g], lane);
    warp_store_state(&fin_start[g], st, lane);
    __syncwarp();
    const uint64_t h = rng_hash(seed, (uint64_t)(d.game_base + g), counter, 0x0fe11ULL);
    warp_new_opening(st, d.n, sym ? sym[g] : (int)(h & 7), adj ? adj[g] : (int)((h >> 3) & 1), lane);
    warp_fresh_game(d, g, st, lane);
}

// ---- root read-backs ---------------------------------------------------------------------

__global__ void __launch_bounds__(32 * WPB) k_root_table(TzDev d, int stride, int* out_n, uint16_t* moves,
                                                         uint32_t* visits, uint32_t* eval_tag, uint32_t* eval_bits,
                                                         float* logit, float* prob, float* std_dev) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    const GameTree t = game_tree(d.arena, g);
    int n = (int)tz_meta_nchild(t.meta[0]);
    const uint32_t first = t.first[0];
    if (lane == 0) out_n[g] = n;
    if (n > stride) n = stride;
    for (int i = lane; i < n; i += 32) {
        const uint32_t c = first + i;
        const size_t o = (size_t)g * stride + i;
        const uint32_t m = t.meta[c];
        moves[o] = (uint16_t)tz_meta_move(m);
        visits[o] = t.visits[c];
        eval_tag[o] = tz_meta_tag(m);
        eval_bits[o] = t.eval[c];
        logit[o] = t.logit[c];
        prob[o] = t.prob[c];
        std_dev[o] = t.std_dev[c];
    }
    for (int i = n + lane; i < stride; i += 32) {  // cells past the last child read as zero
        const size_t o = (size_t)g * stride + i;
        moves[o] = 0;
        visits[o] = 0;
        eval_tag[o] = 0;
        eval_bits[o] = 0;
        logit[o] = 0.0f;
        prob[o] = 0.0f;
        std_dev[o] = 0.0f;
    }
}

// per game: {eval tag, eval bits, visits, std bits, child count, arena slots in use}
__global__ void k_root_stats(TzDev d, uint32_t* out) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= d.G) return;
    const GameTree t = game_tree(d.arena, g);
    const uint32_t m = t.meta[0];
    uint32_t* o = out + (size_t)g * 6;
    o[0] = tz_meta_tag(m);
    o[1] = t.eval[0];
    o[2] = t.visits[0];
    o[3] = __float_as_uint(t.std_dev[0]);
    o[4] = tz_meta_nchild(m);
    o[5] = d.arena.next_slot[g];
}

// improved policy (policy.rs:23-48) and UBE target (node/mod.rs:215-230) of every root.
// visitations < 0 selects `most_visited_count()` per root (reanalyze/src/main.rs:196-202).
__global__ void __launch_bounds__(32 * WPB) k_targets(TzDev d, float visitations, float beta, int stride,
                                                      float* out_policy, float* out_ube, int* out_n,
                                                      uint16_t* out_moves) {
    __shared__ float s_p[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    const GameTree t = game_tree(d.arena, g);
    const uint32_t meta = t.meta[0];
    const int n = (int)tz_meta_nchild(meta);
    const uint32_t first = t.first[0];
    const Ev root_ev = ev_make(tz_meta_tag(meta), t.eval[0]);
    float* p = s_p[warp];
    float v = visitations;
    if (v < 0.0f) {
        uint32_t mx = 0;
        for (int i = lane; i < n; i += 32) mx = max(mx, t.visits[first + i]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(FULL_MASK, mx, o));
        v = (float)mx;
    }
    const float root_v = fsqrt(v);
    const float root_q = ev_notnan(root_ev);
    // ube: LAST child maximising -eval + std * beta
    float best = 0.0f;
    int best_i = -1;
    for (int i = lane; i < n; i += 32) {
        const uint32_t c = first + i;
        const uint32_t cm = t.meta[c];
        const Ev e = ev_make(tz_meta_tag(cm), t.eval[c]);
        const bool needs_init = tz_meta_nchild(cm) == 0 && e.tag == TZ_E_VALUE;
        const float sd = t.std_dev[c];
        const float cq = needs_init ? root_q : ev_notnan(ev_negate(e));
        // sigma_improve(q, std, 0.0, v) + logit
        p[i] = fadd(fmul(fadd(cq, fmul(sd, 0.0f)), root_v), t.logit[c]);
        const float key = fadd(ev_notnan(ev_negate(e)), fmul(sd, beta));
        if (best_i < 0 || !(key < best)) {
            best = key;
            best_i = i;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ok = __shfl_xor_sync(FULL_MASK, best, o);
        const int oi = __shfl_xor_sync(FULL_MASK, best_i, o);
        if (oi >= 0 && (best_i < 0 || ok > best || (ok == best && oi > best_i))) {
            best = ok;
            best_i = oi;
        }
    }
    __syncwarp();
    if (!warp_softmax_inplace(p, n, lane)) flag_error(d, TZ_ERR_NAN, lane);
    const int m = n < stride ? n : stride;
    for (int i = lane; i < m; i += 32) {
        out_policy[(size_t)g * stride + i] = p[i];
        if (out_moves) out_moves[(size_t)g * stride + i] = (uint16_t)tz_meta_move(t.meta[first + i]);
    }
    for (int i = m + lane; i < stride; i += 32) {
        out_policy[(size_t)g * stride + i] = 0.0f;
        if (out_moves) out_moves[(size_t)g * stride + i] = 0;
    }
    if (lane == 0) {
        out_n[g] = n;
        float ube = 0.0f;
        if (!ev_known(root_ev) && n > 0) {
            const float sd = t.std_dev[first + best_i];
            ube = fmul(sd, sd);
        }
        out_ube[g] = ube;
    }
}

// value target of `reanalyze` (reanalyze/src/main.rs:184-195): the root's evaluation when it is known, else the negated
// evaluation of the child the search selected; as f32 (eval.rs:95-105)
__global__ void __launch_bounds__(32 * WPB) k_reanalyze_values(TzDev d, const uint16_t* selected, float* out_value) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    const GameTree t = game_tree(d.arena, g);
    const uint32_t meta = t.meta[0];
    const Ev root_ev = ev_make(tz_meta_tag(meta), t.eval[0]);
    if (ev_known(root_ev)) {
        if (lane == 0) out_value[g] = ev_to_f32(root_ev);
        return;
    }
    const int n = (int)tz_meta_nchild(meta);
    const uint32_t first = t.first[0];
    const uint16_t mv = selected[g];
    int found = 0x7fffffff;
    for (int i = lane; i < n; i += 32)
        if (tz_meta_move(t.meta[first + i]) == mv && i < found) found = i;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) found = min(found, __shfl_xor_sync(FULL_MASK, found, o));
    if (found == 0x7fffffff) {  // "all non-terminal nodes should have at least one child"
        flag_error(d, TZ_ERR_NO_CHILD, lane);
        if (lane == 0) out_value[g] = 0.0f;
        return;
    }
    if (lane == 0) out_value[g] = ev_to_f32(ev_negate(node_eval(t, first + (uint32_t)found)));
}

// select_best_action (node/mod.rs:132-163) of node `slot`; returns the child index, -1 without children
__device__ __forceinline__ int warp_select_best(const GameTree& t, int lane, uint32_t slot = 0) {
    const uint32_t meta = t.meta[slot];
    const int n = (int)tz_meta_nchild(meta);
    const uint32_t first = t.first[slot];
    if (n == 0) return -1;
    if (tz_meta_tag(meta) != TZ_E_VALUE) {
        Ev m;
        return warp_min_child(t, first, n, lane, &m);
    }
    // last maximum of visits, else last maximum of probability
    uint32_t bv = 0;
    int bvi = -1;
    float bp = 0.0f;
    int bpi = -1;
    for (int i = lane; i < n; i += 32) {
        const uint32_t vis = t.visits[first + i];
        const float pr = t.prob[first + i];
        if (bvi < 0 || vis >= bv) {
            bv = vis;
            bvi = i;
        }
        if (bpi < 0 || !(pr < bp)) {
            bp = pr;
            bpi = i;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const uint32_t ov = __shfl_xor_sync(FULL_MASK, bv, o);
        const int ovi = __shfl_xor_sync(FULL_MASK, bvi, o);
        if (ovi >= 0 && (bvi < 0 || ov > bv || (ov == bv && ovi > bvi))) {
            bv = ov;
            bvi = ovi;
        }
        const float op = __shfl_xor_sync(FULL_MASK, bp, o);
        const int opi = __shfl_xor_sync(FULL_MASK, bpi, o);
        if (opi >= 0 && (bpi < 0 || op > bp || (op == bp && opi > bpi))) {
            bp = op;
            bpi = opi;
        }
    }
    return bv == 0 ? bpi : bvi;
}

// select_best_actions / select_actions_in_selfplay (batched.rs:152-183, node/mod.rs:170-207).
// `randoms` replaces the `rand` draw of choose_weighted: the sampled child is the first
// whose cumulative weight exceeds randoms[g] % total (same rule as the oracle).
__global__ void __launch_bounds__(32 * WPB) k_select_actions(TzDev d, int weighted_random_plies, uint32_t threshold,
                                                             float allowed_drop, const unsigned long long* randoms,
                                                             unsigned long long seed, unsigned long long counter,
                                                             uint16_t* out_moves) {
    __shared__ uint32_t s_w[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    const GameTree t = game_tree(d.arena, g);
    const uint32_t meta = t.meta[0];
    const int n = (int)tz_meta_nchild(meta);
    const uint32_t first = t.first[0];
    if (n == 0) {
        if (!(tz_meta_tag(meta) != TZ_E_VALUE && t.eval[0] == 0)) flag_error(d, TZ_ERR_NO_CHILD, lane);
        if (lane == 0) out_moves[g] = 0xffff;
        return;
    }
    int pick = -1;
    const bool sample = tz_meta_tag(meta) == TZ_E_VALUE && (int)d.env[g].ply < weighted_random_plies;
    if (sample) {
        Ev best_eval;
        warp_min_child(t, first, n, lane, &best_eval);
        Ev limit = best_eval;
        if (limit.tag == TZ_E_VALUE) limit.bits = __float_as_uint(fadd(__uint_as_float(limit.bits), allowed_drop));
        uint32_t* w = s_w[warp];
        unsigned long long part = 0;
        for (int i = lane; i < n; i += 32) {
            const uint32_t c = first + i;
            const Ev e = node_eval(t, c);
            const uint32_t vis = t.visits[c];
            const bool drop = vis < threshold || e.tag == TZ_E_WIN || ev_cmp(e, limit) > 0;
            w[i] = drop ? 0u : vis;
            part += w[i];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(FULL_MASK, part, o);
        __syncwarp();
        if (part > 0) {
            const unsigned long long r =
                randoms ? randoms[g] : rng_hash(seed, (uint64_t)(d.game_base + g), counter, 0x5e1ecULL);
            if (lane == 0) {
                unsigned long long x = r % part;
                for (int i = 0; i < n; i++) {
                    if (w[i] == 0) continue;
                    if (x < w[i]) {
                        pick = i;
                        break;
                    }
                    x -= w[i];
                }
            }
            pick = __shfl_sync(FULL_MASK, pick, 0);
        }
    }
    if (pick < 0) pick = warp_select_best(t, lane);
    if (lane == 0) out_moves[g] = (uint16_t)tz_meta_move(t.meta[first + (uint32_t)pick]);
}

// selfplay/src/main.rs:143-152: plies below WEIGHTED_RANDOM_PLIES take the sampled action
__global__ void k_merge_moves(TzDev d, int weighted_random_plies, const uint16_t* sampled, uint16_t* moves) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= d.G) return;
    if ((int)d.env[g].ply < weighted_random_plies) moves[g] = sampled[g];
}

// Node::principal_variation (node/mod.rs:40-62), one warp per tree: game d.tree_game[t] -> out_moves[t][cap], out_len[t]
__global__ void __launch_bounds__(32) k_tree_pv(TzDev d, uint16_t* out_moves, int cap, int* out_len) {
    const int lane = threadIdx.x & 31;
    const GameTree t = game_tree(d.arena, d.tree_game[blockIdx.x]);
    out_moves += (size_t)blockIdx.x * cap;
    out_len += blockIdx.x;
    uint32_t slot = 0;
    int len = 0;
    while (len < cap) {
        const uint32_t meta = t.meta[slot];
        const uint32_t tag = tz_meta_tag(meta);
        const bool needs_init = tz_meta_nchild(meta) == 0 && tag == TZ_E_VALUE;
        const bool terminal = tag != TZ_E_VALUE && t.eval[slot] == 0;
        if (needs_init || terminal) break;
        const int idx = warp_select_best(t, lane, slot);
        if (idx < 0) break;
        slot = t.first[slot] + (uint32_t)idx;
        if (lane == 0) out_moves[len] = (uint16_t)tz_meta_move(t.meta[slot]);
        len++;
    }
    if (lane == 0) *out_len = len;
}

// overwrite the priors of every root's children (Node::apply_dirichlet, node/noise.rs:10-26: the mixing and
// the `ln` are done by the host with its libm, like the reference; this only stores the result)
__global__ void __launch_bounds__(32 * WPB) k_set_root_priors(TzDev d, int stride, const float* prob, const float* logit) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    const GameTree t = game_tree(d.arena, g);
    int n = (int)tz_meta_nchild(t.meta[0]);
    if (n > stride) n = stride;
    const uint32_t first = t.first[0];
    bool bad = false;
    for (int i = lane; i < n; i += 32) {
        const float p = prob[(size_t)g * stride + i], l = logit[(size_t)g * stride + i];
        if (p != p || l != l || p < 0.0f) {  // NotNan in the reference; -inf logits (ln 0) are fine
            bad = true;
            continue;
        }
        t.prob[first + i] = p;
        t.logit[first + i] = l;
    }
    if (__any_sync(FULL_MASK, bad)) flag_error(d, TZ_ERR_NAN, lane);
}

// ---- rules parity hooks --------------------------------------------------------------------

__global__ void __launch_bounds__(32 * WPB) k_rules_probe(TzDev d, const TzState* states, int count, int stride,
                                                          uint16_t* out_moves, int* out_n, int* out_terminal,
                                                          int* out_result) {
    __shared__ TzState s_state[WPB];
    __shared__ uint16_t s_moves[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * WPB + warp;
    if (i >= count) return;
    TzState* st = &s_state[warp];
    warp_load_state(st, &states[i], lane);
    if (out_terminal) {
        const int term = warp_terminal(st, d.n, d.half_komi, d.rev_limit, lane);
        if (lane == 0) out_terminal[i] = term;
    }
    if (out_result) {
        const int res = warp_game_result(st, d.n, d.half_komi, d.rev_limit, lane);
        if (lane == 0) out_result[i] = res;
    }
    if (out_moves) {
        const int cnt = warp_movegen(st, d.n, s_moves[warp], lane);
        if (lane == 0) out_n[i] = cnt;
        const int m = cnt < stride ? cnt : stride;
        for (int j = lane; j < m; j += 32) out_moves[(size_t)i * stride + j] = s_moves[warp][j];
    }
}

__global__ void __launch_bounds__(32 * WPB) k_apply_moves(TzDev d, TzState* states, const uint16_t* moves, int count,
                                                          int* out_ok) {
    __shared__ TzState s_state[WPB];
    __shared__ uint16_t s_moves[WPB][TZ_MAX_MOVES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * WPB + warp;
    if (i >= count) return;
    TzState* st = &s_state[warp];
    warp_load_state(st, &states[i], lane);
    const bool ok = warp_apply_checked(st, d.n, moves[i], s_moves[warp], lane);
    if (ok) warp_store_state(&states[i], st, lane);
    if (lane == 0 && out_ok) out_ok[i] = ok ? 1 : 0;
}

// parity hook: the device's expf (tree.cuh `expf_libm`, the softmax's exp) on arbitrary inputs
__global__ void k_debug_expf(const float* in, int count, float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = expf_libm(in[i]);
}

// ---- resident self-play training data (selfplay/src/main.rs:238-329 on the device) ------------------

__device__ __forceinline__ uint32_t record_bytes(int n) {
    return (uint32_t)sizeof(TzRecHead) + (((uint32_t)n * 6u + 15u) & ~15u);
}

// selfplay/src/main.rs:173: the exploration half keeps only targets past the weighted-random plies
__device__ __forceinline__ bool record_kept(int g, int exploration_games, int ply, int weighted_random_plies) {
    return g >= exploration_games || ply > weighted_random_plies;
}

// take_a_step (main.rs:238-258): append one pending record per game -- the root position, its replay index, the
// improved policy / UBE target k_targets left in `policy` [G][stride] / `ube` / `tbl_n`, the root's moves in child
// order.  A game whose region is full records nothing more until it ends.
__global__ void __launch_bounds__(32 * WPB) k_record(TzDev d, TzRecorder r, const float* policy, const float* ube,
                                                     const int* tbl_n, int stride) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G || r.full[g]) return;
    int n = tbl_n[g];
    if (n > stride) n = stride;
    const uint32_t size = record_bytes(n);
    const uint32_t cnt = r.count[g], used = r.used[g];
    if (cnt >= TZ_MAX_PLIES || (unsigned long long)used + size > r.bytes_per_game) {
        if (lane == 0) {
            r.full[g] = 1;
            atomicOr(d.status, TZ_ERR_TARGETS_FULL);
        }
        return;
    }
    unsigned char* rec = r.store + (size_t)g * r.bytes_per_game + used;
    TzRecHead* head = reinterpret_cast<TzRecHead*>(rec);
    warp_load_state(&head->env, &d.env[g], lane);
    if (lane == 0) {
        head->p = d.replay_len[g];
        head->n = n;
        head->ube = ube[g];
        head->pad = 0;
    }
    float* probs = reinterpret_cast<float*>(rec + sizeof(TzRecHead));
    uint16_t* moves = reinterpret_cast<uint16_t*>(probs + n);
    const GameTree t = game_tree(d.arena, g);
    const uint32_t first = t.first[0];
    for (int i = lane; i < n; i += 32) {
        probs[i] = policy[(size_t)g * stride + i];
        moves[i] = (uint16_t)tz_meta_move(t.meta[first + i]);
    }
    if (lane == 0) {
        r.rec_off[(size_t)g * TZ_MAX_PLIES + cnt] = used;
        r.count[g] = cnt + 1;
        r.used[g] = used + size;
        atomicMax(r.high_water, used + size);
    }
}

// what every game k_restart finished emits: kept targets, their policy entries, one replay, its moves
__global__ void __launch_bounds__(32 * WPB) k_emit_count(TzDev d, TzRecorder r, const int* terminal, const int* fin_len,
                                                         int weighted_random_plies, int exploration_games) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    unsigned long long* c = r.g_count + (size_t)g * TZ_Q_KINDS;
    if (terminal[g] == TZ_T_NONE) {
        if (lane < TZ_Q_KINDS) c[lane] = 0;
        return;
    }
    const int cnt = (int)r.count[g];
    const unsigned char* region = r.store + (size_t)g * r.bytes_per_game;
    unsigned long long kept = 0, entries = 0;
    for (int j = lane; j < cnt; j += 32) {
        const TzRecHead* h = reinterpret_cast<const TzRecHead*>(region + r.rec_off[(size_t)g * TZ_MAX_PLIES + j]);
        if (record_kept(g, exploration_games, (int)h->env.ply, weighted_random_plies)) {
            kept++;
            entries += (unsigned long long)h->n;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        kept += __shfl_xor_sync(FULL_MASK, kept, o);
        entries += __shfl_xor_sync(FULL_MASK, entries, o);
    }
    if (lane == 0) {
        c[TZ_Q_TARGETS] = kept;
        c[TZ_Q_POLICY] = entries;
        c[TZ_Q_REPLAYS] = 1;
        c[TZ_Q_MOVES] = (unsigned long long)fin_len[g];
    }
}

// exclusive scan of the per-game counts over games in index order (one block): game g's data goes to
// fill + (sum over games < g).  The games that fit form a prefix (the sums only grow); the first game that does not
// fit and every later one are dropped (their records are lost), TZ_ERR_TARGETS_FULL is raised, and the queue fill
// advances past the games that fit only.
__global__ void __launch_bounds__(1024) k_emit_scan(TzDev d, TzRecorder r) {
    __shared__ unsigned long long s_warp[32][TZ_Q_KINDS];
    __shared__ unsigned long long s_carry[TZ_Q_KINDS], s_fill[TZ_Q_KINDS];
    __shared__ int s_dropped;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < TZ_Q_KINDS) {
        s_carry[tid] = 0;
        s_fill[tid] = r.fill[tid];
    }
    if (tid == 0) s_dropped = 0;
    __syncthreads();
    for (int base = 0; base < d.G; base += 1024) {
        const int g = base + tid;
        unsigned long long v[TZ_Q_KINDS], incl[TZ_Q_KINDS];
#pragma unroll
        for (int q = 0; q < TZ_Q_KINDS; q++) {
            v[q] = g < d.G ? r.g_count[(size_t)g * TZ_Q_KINDS + q] : 0ull;
            incl[q] = v[q];
        }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
#pragma unroll
            for (int q = 0; q < TZ_Q_KINDS; q++) {
                const unsigned long long y = __shfl_up_sync(FULL_MASK, incl[q], o);
                if (lane >= o) incl[q] += y;
            }
        if (lane == 31)
            for (int q = 0; q < TZ_Q_KINDS; q++) s_warp[warp][q] = incl[q];
        __syncthreads();
        if (warp == 0) {
#pragma unroll
            for (int q = 0; q < TZ_Q_KINDS; q++) {
                unsigned long long x = s_warp[lane][q];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned long long y = __shfl_up_sync(FULL_MASK, x, o);
                    if (lane >= o) x += y;
                }
                s_warp[lane][q] = x;
            }
        }
        __syncthreads();
        if (g < d.G && v[TZ_Q_REPLAYS] != 0) {
            unsigned long long at[TZ_Q_KINDS];
            bool fits = true;
#pragma unroll
            for (int q = 0; q < TZ_Q_KINDS; q++) {
                const unsigned long long before = s_carry[q] + (warp ? s_warp[warp - 1][q] : 0ull) + incl[q] - v[q];
                at[q] = r.fill[q] + before;
                fits = fits && at[q] + v[q] <= r.cap[q];
            }
            unsigned long long* b = r.g_base + (size_t)g * TZ_Q_KINDS;
            if (fits) {
#pragma unroll
                for (int q = 0; q < TZ_Q_KINDS; q++) {
                    b[q] = at[q];
                    atomicMax(&s_fill[q], at[q] + v[q]);
                }
            } else {
                b[0] = ~0ull;
                s_dropped = 1;
            }
        }
        __syncthreads();
        if (tid < TZ_Q_KINDS) s_carry[tid] += s_warp[31][tid];
        __syncthreads();
    }
    if (tid < TZ_Q_KINDS) r.fill[tid] = s_fill[tid];
    if (tid == 0 && s_dropped) atomicOr(d.status, TZ_ERR_TARGETS_FULL);
}

// restart_envs_and_complete_targets (main.rs:263-329): the finished game's replay, then its targets from the last ply
// to the first with value = Eval::from(terminal) negated L - p times (L = replay length, p = the record's replay
// index), the exploration half filtered by ply; every finished game's cursor is reset
__global__ void __launch_bounds__(32 * WPB) k_emit_write(TzDev d, TzRecorder r, const int* terminal, const int* fin_len,
                                                         const TzState* fin_start, const uint16_t* fin_replay,
                                                         int weighted_random_plies, int exploration_games) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * WPB + warp;
    if (g >= d.G) return;
    const int term = terminal[g];
    if (term == TZ_T_NONE) return;
    const unsigned long long* b = r.g_base + (size_t)g * TZ_Q_KINDS;
    if (b[TZ_Q_TARGETS] != ~0ull) {
        const unsigned long long ri = b[TZ_Q_REPLAYS], mo = b[TZ_Q_MOVES];
        const int L = fin_len[g];
        warp_load_state(&r.r_start[ri], &fin_start[g], lane);
        if (lane == 0) {
            r.r_result[ri] = r.result[g];
            r.r_terminal[ri] = term;
            r.r_len[ri] = L;
            r.r_off[ri] = mo;
            r.r_game[ri] = d.game_base + g;
            r.r_exploration[ri] = g < exploration_games ? 1 : 0;
        }
        for (int i = lane; i < L; i += 32) r.r_moves[mo + i] = fin_replay[(size_t)g * TZ_MAX_PLIES + i];
        unsigned long long ti = b[TZ_Q_TARGETS], po = b[TZ_Q_POLICY];
        const unsigned char* region = r.store + (size_t)g * r.bytes_per_game;
        Ev e = ev_from_terminal(term);
        int pc = L;
        for (int j = (int)r.count[g] - 1; j >= 0; j--) {
            const unsigned char* rec = region + r.rec_off[(size_t)g * TZ_MAX_PLIES + j];
            const TzRecHead* h = reinterpret_cast<const TzRecHead*>(rec);
            const int p = h->p, n = h->n;
            for (; pc > p; pc--) e = ev_negate(e);
            if (!record_kept(g, exploration_games, (int)h->env.ply, weighted_random_plies)) continue;
            warp_load_state(&r.t_env[ti], &h->env, lane);
            if (lane == 0) {
                r.t_value[ti] = ev_to_f32(e);
                r.t_ube[ti] = h->ube;
                r.t_n[ti] = n;
                r.t_off[ti] = po;
                r.t_game[ti] = d.game_base + g;
            }
            const float* probs = reinterpret_cast<const float*>(rec + sizeof(TzRecHead));
            const uint16_t* moves = reinterpret_cast<const uint16_t*>(probs + n);
            for (int i = lane; i < n; i += 32) {
                r.p_probs[po + i] = probs[i];
                r.p_moves[po + i] = moves[i];
            }
            ti++;
            po += (unsigned long long)n;
        }
    }
    __syncwarp();
    if (lane == 0) {
        r.count[g] = 0;
        r.used[g] = 0;
        r.full[g] = 0;
    }
}

// ---- launchers -------------------------------------------------------------------------------

static inline int blocks_for(int items) { return (items + WPB - 1) / WPB; }

void launch_record(const TzDev& d, const TzRecorder& r, const float* policy, const float* ube, const int* n, int stride,
                   cudaStream_t st) {
    k_record<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, r, policy, ube, n, stride);
}
void launch_emit(const TzDev& d, const TzRecorder& r, const int* terminal, const int* fin_len, const TzState* fin_start,
                 const uint16_t* fin_replay, int weighted_random_plies, int exploration_games, cudaStream_t st) {
    k_emit_count<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, r, terminal, fin_len, weighted_random_plies, exploration_games);
    k_emit_scan<<<1, 1024, 0, st>>>(d, r);
    k_emit_write<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, r, terminal, fin_len, fin_start, fin_replay,
                                                       weighted_random_plies, exploration_games);
}

void launch_select(const TzDev& d, int phase, int halving_i, const float* betas, cudaStream_t st) {
    k_select<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, phase, halving_i, betas);
}
void launch_agent_synth(const TzDev& d, cudaStream_t st) { k_agent_synth<<<blocks_for(d.Q), 32 * WPB, 0, st>>>(d); }
void launch_expand(const TzDev& d, cudaStream_t st) { k_expand<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d); }
void launch_gumbel_noise(const TzDev& d, float* out, int stride, unsigned long long seed, unsigned long long counter,
                         cudaStream_t st) {
    const size_t total = (size_t)d.G * stride;
    k_gumbel_noise<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d, out, stride, seed, counter);
}
void launch_gumbel_init(const TzDev& d, int k, const float* gumbel, int stride, cudaStream_t st) {
    k_gumbel_init<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, k, gumbel, stride);
}
void launch_halve(const TzDev& d, const float* betas, float visits, int remaining, cudaStream_t st) {
    k_halve<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, betas, visits, remaining);
}
void launch_finalize(const TzDev& d, uint16_t* out_moves, cudaStream_t st) {
    k_finalize<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, out_moves);
}
void launch_step(const TzDev& d, const uint16_t* moves, cudaStream_t st, const uint8_t* mask) {
    k_step<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, moves, mask);
}
static int tree_warps(int warps) { return warps >= 1 && warps <= TREE_WARPS ? warps : TREE_WARPS; }

void launch_tree_forward(const TzDev& d, int trees, float beta, int batch_size, int max_forwards, int warps,
                         cudaStream_t st) {
    static const cudaError_t attr = cudaFuncSetAttribute(k_tree_forward, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                        (int)sizeof(TreeForwardSmem));
    (void)attr;
    k_tree_forward<<<trees, 32 * tree_warps(warps), sizeof(TreeForwardSmem), st>>>(d, beta, batch_size, max_forwards);
}
void launch_tree_backward(const TzDev& d, int trees, int batch_size, int warps, cudaStream_t st) {
    static const cudaError_t attr = cudaFuncSetAttribute(k_tree_backward, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                        (int)sizeof(TreeBackwardSmem));
    (void)attr;
    k_tree_backward<<<trees, 32 * tree_warps(warps), sizeof(TreeBackwardSmem), st>>>(d, batch_size);
}
void launch_set_root_priors(const TzDev& d, int stride, const float* prob, const float* logit, cudaStream_t st) {
    k_set_root_priors<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, stride, prob, logit);
}
void launch_tree_pv(const TzDev& d, int trees, uint16_t* out_moves, int cap, int* out_len, cudaStream_t st) {
    k_tree_pv<<<trees, 32, 0, st>>>(d, out_moves, cap, out_len);
}
void launch_new_openings(const TzDev& d, const uint8_t* mask, const int* sym, const int* adj, unsigned long long seed,
                         unsigned long long counter, cudaStream_t st) {
    k_new_openings<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, mask, sym, adj, seed, counter);
}
void launch_random_steps(const TzDev& d, const uint8_t* mask, int steps, unsigned long long seed, cudaStream_t st) {
    k_random_steps<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, mask, steps, seed);
}
void launch_set_positions(const TzDev& d, const TzState* states, const uint8_t* mask, cudaStream_t st) {
    k_set_positions<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, states, mask);
}
void launch_gather_positions(const TzDev& d, const TzState* pool, const uint32_t* indices, cudaStream_t st) {
    k_gather_positions<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, pool, indices);
}
void launch_reanalyze_values(const TzDev& d, const uint16_t* selected, float* out_value, cudaStream_t st) {
    k_reanalyze_values<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, selected, out_value);
}
void launch_reset_roots(const TzDev& d, const uint8_t* mask, cudaStream_t st) {
    k_reset_roots<<<(d.G + 127) / 128, 128, 0, st>>>(d, mask);
}
void launch_restart(const TzDev& d, const int* sym, const int* adj, unsigned long long seed, unsigned long long counter,
                    int* out_terminal, TzState* fin_start, uint16_t* fin_replay, int* fin_len, cudaStream_t st,
                    int* out_result) {
    k_restart<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, sym, adj, seed, counter, out_terminal, fin_start, fin_replay,
                                                    fin_len, out_result);
}
void launch_root_table(const TzDev& d, int stride, int* out_n, uint16_t* moves, uint32_t* visits, uint32_t* eval_tag,
                       uint32_t* eval_bits, float* logit, float* prob, float* std_dev, cudaStream_t st) {
    k_root_table<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, stride, out_n, moves, visits, eval_tag, eval_bits, logit, prob,
                                                       std_dev);
}
void launch_root_stats(const TzDev& d, uint32_t* out, cudaStream_t st) {
    k_root_stats<<<(d.G + 127) / 128, 128, 0, st>>>(d, out);
}
void launch_targets(const TzDev& d, float visitations, float beta, int stride, float* out_policy, float* out_ube,
                    int* out_n, uint16_t* out_moves, cudaStream_t st) {
    k_targets<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, visitations, beta, stride, out_policy, out_ube, out_n, out_moves);
}
void launch_select_actions(const TzDev& d, int weighted_random_plies, uint32_t threshold, float allowed_drop,
                           const unsigned long long* randoms, unsigned long long seed, unsigned long long counter,
                           uint16_t* out_moves, cudaStream_t st) {
    k_select_actions<<<blocks_for(d.G), 32 * WPB, 0, st>>>(d, weighted_random_plies, threshold, allowed_drop, randoms,
                                                           seed, counter, out_moves);
}
void launch_merge_moves(const TzDev& d, int weighted_random_plies, const uint16_t* sampled, uint16_t* moves,
                        cudaStream_t st) {
    k_merge_moves<<<(d.G + 127) / 128, 128, 0, st>>>(d, weighted_random_plies, sampled, moves);
}
void launch_debug_expf(const float* in, int count, float* out, cudaStream_t st) {
    k_debug_expf<<<(count + 255) / 256, 256, 0, st>>>(in, count, out);
}
void launch_rules_probe(const TzDev& d, const TzState* states, int count, int stride, uint16_t* out_moves, int* out_n,
                        int* out_terminal, int* out_result, cudaStream_t st) {
    k_rules_probe<<<blocks_for(count), 32 * WPB, 0, st>>>(d, states, count, stride, out_moves, out_n, out_terminal,
                                                          out_result);
}
void launch_apply_moves(const TzDev& d, TzState* states, const uint16_t* moves, int count, int* out_ok,
                        cudaStream_t st) {
    k_apply_moves<<<blocks_for(count), 32 * WPB, 0, st>>>(d, states, moves, count, out_ok);
}
