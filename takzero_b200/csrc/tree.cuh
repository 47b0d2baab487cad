// tree.cuh -- Eval arithmetic and exact-f32 helpers for the tree kernels (sm_100a).
//
// Every expression that feeds a comparison in the reference's search is evaluated
// here in the reference's order in IEEE binary32 with explicit round-to-nearest
// intrinsics (never contracted into FMA), see SURVEY App. A.8:
//   eval.rs:40-47,95-105,138-163   negate / f32::from / Ord
//   policy.rs:10-19                softmax (libm expf, restated below bit for bit)
//   policy.rs:140-156              exploration_rate / PUCT
#pragma once
#include "common.cuh"

struct Ev {
    uint32_t tag;
    uint32_t bits;  // f32 bits for TZ_E_VALUE, ply otherwise
};

__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float fsqrt(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ float fneg(float a) { return __uint_as_float(__float_as_uint(a) ^ 0x80000000u); }

__device__ __forceinline__ Ev ev_make(uint32_t tag, uint32_t bits) {
    Ev e;
    e.tag = tag;
    e.bits = bits;
    return e;
}
__device__ __forceinline__ Ev ev_value(float v) { return ev_make(TZ_E_VALUE, __float_as_uint(v)); }
__device__ __forceinline__ bool ev_known(Ev e) { return e.tag != TZ_E_VALUE; }

__device__ __forceinline__ Ev ev_negate(Ev e) {  // eval.rs:40-47
    switch (e.tag) {
        case TZ_E_VALUE: return ev_value(fneg(__uint_as_float(e.bits)));
        case TZ_E_WIN: return ev_make(TZ_E_LOSS, e.bits + 1);
        case TZ_E_DRAW: return ev_make(TZ_E_DRAW, e.bits + 1);
        default: return ev_make(TZ_E_WIN, e.bits + 1);
    }
}

// Eval::from(terminal) (eval.rs:118-126): tz_result codes 1 win, 2 loss, 3 draw are the tags Win / Loss / Draw at ply 0
__device__ __forceinline__ Ev ev_from_terminal(int terminal) { return ev_make((uint32_t)terminal, 0u); }

// compiler-rt __powisf2(0.997f, ply): what Rust's f32::powi lowers to (eval.rs:97)
__device__ __forceinline__ float powi_discount(int b) {
    float a = 0.997f, r = 1.0f;
    while (true) {
        if (b & 1) r = fmul(r, a);
        b >>= 1;
        if (b == 0) break;
        a = fmul(a, a);
    }
    return r;
}

__device__ __forceinline__ float ev_to_f32(Ev e) {  // eval.rs:95-105
    if (e.tag == TZ_E_VALUE) return fmul(1.0f, __uint_as_float(e.bits));
    const float m = e.tag == TZ_E_WIN ? 1.0f : (e.tag == TZ_E_LOSS ? -1.0f : 0.0f);
    return fmul(powi_discount((int)e.bits), m);
}

__device__ __forceinline__ float ev_notnan(Ev e) {  // eval.rs:107-116
    return e.tag == TZ_E_VALUE ? __uint_as_float(e.bits) : ev_to_f32(e);
}

__device__ __forceinline__ int cmp_f(float a, float b) { return (a > b) - (a < b); }
__device__ __forceinline__ int cmp_u(uint32_t a, uint32_t b) { return (a > b) - (a < b); }

__device__ __forceinline__ int ev_cmp(Ev a, Ev b) {  // eval.rs:138-163, CONTEMPT = -0.05
    const float contempt = -0.05f;
    switch (a.tag) {
        case TZ_E_VALUE:
            switch (b.tag) {
                case TZ_E_VALUE: return cmp_f(__uint_as_float(a.bits), __uint_as_float(b.bits));
                case TZ_E_WIN: return -1;
                case TZ_E_DRAW: return cmp_f(__uint_as_float(a.bits), contempt);
                default: return 1;
            }
        case TZ_E_WIN: return b.tag == TZ_E_WIN ? cmp_u(b.bits, a.bits) : 1;
        case TZ_E_DRAW:
            switch (b.tag) {
                case TZ_E_VALUE: return cmp_f(contempt, __uint_as_float(b.bits));
                case TZ_E_WIN: return -1;
                case TZ_E_DRAW: return cmp_u(b.bits, a.bits);
                default: return 1;
            }
        default: return b.tag == TZ_E_LOSS ? cmp_u(a.bits, b.bits) : -1;
    }
}

// glibc 2.39 expf (sysdeps/ieee754/flt-32/e_expf.c, the exp2f_data table algorithm)
// restated in double precision with explicit round-to-nearest ops.  Verified on the
// build host against libm expf for every third binary32 in [-112, 0]: 1 mismatch in
// 1.1e9 (at exp(x) ~ 2^-91).  Rust's f32::exp calls this libm routine on Linux.
__device__ const uint64_t tz_exp2f_tab[32] = {
    0x3ff0000000000000ULL, 0x3fefd9b0d3158574ULL, 0x3fefb5586cf9890fULL, 0x3fef9301d0125b51ULL,
    0x3fef72b83c7d517bULL, 0x3fef54873168b9aaULL, 0x3fef387a6e756238ULL, 0x3fef1e9df51fdee1ULL,
    0x3fef06fe0a31b715ULL, 0x3feef1a7373aa9cbULL, 0x3feedea64c123422ULL, 0x3feece086061892dULL,
    0x3feebfdad5362a27ULL, 0x3feeb42b569d4f82ULL, 0x3feeab07dd485429ULL, 0x3feea47eb03a5585ULL,
    0x3feea09e667f3bcdULL, 0x3fee9f75e8ec5f74ULL, 0x3feea11473eb0187ULL, 0x3feea589994cce13ULL,
    0x3feeace5422aa0dbULL, 0x3feeb737b0cdc5e5ULL, 0x3feec49182a3f090ULL, 0x3feed503b23e255dULL,
    0x3feee89f995ad3adULL, 0x3feeff76f2fb5e47ULL, 0x3fef199bdd85529cULL, 0x3fef3720dcef9069ULL,
    0x3fef5818dcfba487ULL, 0x3fef7c97337b9b5fULL, 0x3fefa4afa2a490daULL, 0x3fefd0765b6e4540ULL};

__device__ __forceinline__ float expf_libm(float x) {
    if (x != x) return x;
    if (x > 88.72283172607421875f) return __int_as_float(0x7f800000);  // 0x1.62e42ep6f
    if (x < -103.97207641601562500f) return 0.0f;                      // -0x1.9fe368p6f
    const double N = 32.0;
    const double inv_ln2_n = 0x1.71547652b82fep+0 * N;
    const double c0 = 0x1.c6af84b912394p-5 / N / N / N;
    const double c1 = 0x1.ebfce50fac4f3p-3 / N / N;
    const double c2 = 0x1.62e42ff0c52d6p-1 / N;
    const double shift = 0x1.8p+52;
    const double xd = (double)x;
    double z = __dmul_rn(inv_ln2_n, xd);
    double kd = __dadd_rn(z, shift);
    const uint64_t ki = (uint64_t)__double_as_longlong(kd);
    kd = __dsub_rn(kd, shift);
    const double r = __dsub_rn(z, kd);
    uint64_t t = tz_exp2f_tab[ki & 31];
    t += ki << (52 - 5);
    const double s = __longlong_as_double((long long)t);
    z = __dadd_rn(__dmul_rn(c0, r), c1);
    const double r2 = __dmul_rn(r, r);
    double y = __dadd_rn(__dmul_rn(c2, r), 1.0);
    y = __dadd_rn(__dmul_rn(z, r2), y);
    y = __dmul_rn(y, s);
    return __double2float_rn(y);
}

// ---- arena view of one game ------------------------------------------------------

struct GameTree {
    uint32_t* eval;
    uint32_t* meta;
    uint32_t* visits;
    float* prob;
    float* std_dev;
    float* logit;
    uint32_t* first;
};

__device__ __forceinline__ GameTree game_tree_half(const TzArena& a, int g, int half) {
    GameTree t;
    const size_t o = ((size_t)g * 2 + (size_t)half) * a.cap;
    t.eval = a.eval + o;
    t.meta = a.meta + o;
    t.visits = a.visits + o;
    t.prob = a.prob + o;
    t.std_dev = a.std_dev + o;
    t.logit = a.logit + o;
    t.first = a.first + o;
    return t;
}

__device__ __forceinline__ GameTree game_tree(const TzArena& a, int g) {
    return game_tree_half(a, g, a.half[g]);
}

__device__ __forceinline__ Ev node_eval(const GameTree& t, uint32_t slot) {
    return ev_make(tz_meta_tag(t.meta[slot]), t.eval[slot]);
}

// lane 0 only
__device__ __forceinline__ void node_set_eval(const GameTree& t, uint32_t slot, Ev e) {
    const uint32_t m = t.meta[slot];
    t.meta[slot] = (m & ~(3u << 16)) | (e.tag << 16);
    t.eval[slot] = e.bits;
}

// Node::default() (node/mod.rs:25-38) into `slot`; lane 0 only
__device__ __forceinline__ void node_reset(const GameTree& t, uint32_t slot) {
    t.eval[slot] = 0;
    t.meta[slot] = 0;
    t.visits[slot] = 0;
    t.prob[slot] = 0.0f;
    t.std_dev[slot] = 0.0f;
    t.logit[slot] = 0.0f;
    t.first[slot] = 0;
}

// ---- warp reductions --------------------------------------------------------------

// minimum Eval over the children of `slot` in the reference's order (Iterator::min /
// min_by_key keep the FIRST minimum); returns the child index, the eval in *out.
__device__ __forceinline__ int warp_min_child(const GameTree& t, uint32_t first, int nchild, int lane,
                                              Ev* out) {
    Ev best = ev_make(TZ_E_WIN, 0);  // greatest possible
    int best_i = 0x7fffffff;
    for (int i = lane; i < nchild; i += 32) {
        const Ev e = node_eval(t, first + i);
        if (best_i == 0x7fffffff || ev_cmp(e, best) < 0) {
            best = e;
            best_i = i;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Ev oe;
        oe.tag = __shfl_xor_sync(0xffffffffu, best.tag, o);
        oe.bits = __shfl_xor_sync(0xffffffffu, best.bits, o);
        const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
        if (oi != 0x7fffffff) {
            const int c = best_i == 0x7fffffff ? -1 : ev_cmp(oe, best);
            if (best_i == 0x7fffffff || c < 0 || (c == 0 && oi < best_i)) {
                best = oe;
                best_i = oi;
            }
        }
    }
    *out = best;
    return best_i;
}

// children summary used by node_solver (mcts.rs:66-76) and the root recompute
// (batched.rs:381-384): bit 0 = all children known, bit 1 = any child is a loss
__device__ __forceinline__ int warp_children_flags(const GameTree& t, uint32_t first, int nchild,
                                                   int lane) {
    bool all_known = true, any_loss = false;
    for (int i = lane; i < nchild; i += 32) {
        const uint32_t tag = tz_meta_tag(t.meta[first + i]);
        all_known = all_known && tag != TZ_E_VALUE;
        any_loss = any_loss || tag == TZ_E_LOSS;
    }
    const bool ak = __all_sync(0xffffffffu, all_known);
    const bool al = __any_sync(0xffffffffu, any_loss);
    return (ak ? 1 : 0) | (al ? 2 : 0);
}

// ---- selection (policy.rs:78-95) ----------------------------------------------------

__device__ __forceinline__ float exploration_rate(const float* ln_table, uint32_t visits) {
    // ((1 + n + 500) / 500).ln() + 4, tabulated with the host's libm logf for n < TZ_LN_TABLE
    if (visits < TZ_LN_TABLE) return ln_table[visits];
    const float n = (float)visits;
    const float x = fdiv(fadd(fadd(1.0f, n), 500.0f), 500.0f);
    return fadd(__double2float_rn(log((double)x)), 4.0f);
}

// returns the selected child index, or -1 when no child is eligible / a key is NaN
// (`known_visits` >= 0: the caller already holds the node's visit count -- the single-tree wavefront, where a later
// descent may be incrementing it at this very moment)
__device__ __forceinline__ int warp_select_puct(const GameTree& t, uint32_t slot, float beta,
                                                const float* ln_table, int lane, bool* nan_seen,
                                                long long known_visits = -1) {
    const uint32_t meta = t.meta[slot];
    const int nchild = (int)tz_meta_nchild(meta);
    const uint32_t first = t.first[slot];
    const bool parent_is_loss = tz_meta_tag(meta) == TZ_E_LOSS;
    const uint32_t pv = known_visits >= 0 ? (uint32_t)known_visits : t.visits[slot];
    const float parent_visits = (float)pv;
    // exploration_rate(Np) * P * sqrt(Np) / (1 + n): the first and third factors are uniform
    const float rate = exploration_rate(ln_table, pv);
    const float root = fsqrt(parent_visits);
    float best = 0.0f;
    int best_i = -1;
    bool bad = false;
    for (int i = lane; i < nchild; i += 32) {
        const uint32_t c = first + i;
        const Ev e = node_eval(t, c);
        if (!(parent_is_loss || e.tag != TZ_E_WIN)) continue;
        const float q = ev_notnan(ev_negate(e));
        const float puct = fdiv(fmul(fmul(rate, t.prob[c]), root), fadd(1.0f, (float)t.visits[c]));
        const float key = fadd(fadd(q, puct), fmul(t.std_dev[c], beta));
        bad = bad || key != key;
        if (best_i < 0 || !(key < best)) {  // max_by_key keeps the LAST maximum
            best = key;
            best_i = i;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ok = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
        if (oi >= 0 && (best_i < 0 || ok > best || (ok == best && oi > best_i))) {
            best = ok;
            best_i = oi;
        }
    }
    *nan_seen = __any_sync(0xffffffffu, bad);
    return best_i;
}

// ---- backups (mcts.rs:49-102,141-225) -------------------------------------------------

struct Propagated {
    Ev eval;
    float variance;
};

// `propagate_child_eval` on node `slot` (mcts.rs:78-102).  Warp-convergent; lane 0 writes.
__device__ __forceinline__ Propagated warp_propagate(const GameTree& t, uint32_t slot, Propagated child,
                                                     int lane) {
    const uint32_t meta = t.meta[slot];
    const int nchild = (int)tz_meta_nchild(meta);
    const uint32_t first = t.first[slot];
    Ev ev = ev_make(tz_meta_tag(meta), t.eval[slot]);
    float std_dev = t.std_dev[slot];
    // node_solver
    const int flags = warp_children_flags(t, first, nchild, lane);
    if (child.eval.tag == TZ_E_LOSS || (flags & 1)) {
        Ev m;
        warp_min_child(t, first, nchild, lane, &m);
        ev = ev_negate(m);
        std_dev = 0.0f;
        if (lane == 0) {
            node_set_eval(t, slot, ev);
            t.std_dev[slot] = 0.0f;
        }
    }
    Propagated p;
    if (ev_known(ev)) {
        p.eval = ev;
        p.variance = fmul(std_dev, std_dev);
    } else {
        const float negated = ev_notnan(ev_negate(child.eval));
        const float n = (float)t.visits[slot];
        // update_mean_value / update_standard_deviation (evaluation is a Value here)
        float m = __uint_as_float(ev.bits);
        m = fadd(m, fdiv(fadd(fneg(m), negated), n));
        std_dev = fadd(std_dev, fdiv(fadd(fneg(std_dev), fsqrt(child.variance)), n));
        if (lane == 0) {
            t.eval[slot] = __float_as_uint(m);
            t.std_dev[slot] = std_dev;
        }
        p.eval = ev_value(fmul(negated, 0.997f));
        p.variance = fmul(fmul(child.variance, 0.997f), 0.997f);
    }
    __syncwarp();
    return p;
}

// `propagate_child_eval` in two halves for the single-tree wavefront (kernels.cu, k_tree_backward): everything but the
// stores -- same reads, same arithmetic, same order as warp_propagate -- and then the stores.
struct PendingNode {
    uint32_t slot;
    int kind;  // 0 nothing, 1 solved (tag + bits, std_dev 0), 2 running mean (bits, std_dev)
    uint32_t meta, bits;
    float std_dev;
};

__device__ __forceinline__ Propagated warp_propagate_compute(const GameTree& t, uint32_t slot, Propagated child, int lane,
                                                             PendingNode* w) {
    const uint32_t meta = t.meta[slot];
    const int nchild = (int)tz_meta_nchild(meta);
    const uint32_t first = t.first[slot];
    Ev ev = ev_make(tz_meta_tag(meta), t.eval[slot]);
    float std_dev = t.std_dev[slot];
    w->slot = slot;
    w->kind = 0;
    const int flags = warp_children_flags(t, first, nchild, lane);
    if (child.eval.tag == TZ_E_LOSS || (flags & 1)) {
        Ev m;
        warp_min_child(t, first, nchild, lane, &m);
        ev = ev_negate(m);
        std_dev = 0.0f;
        w->kind = 1;
        w->meta = (meta & ~(3u << 16)) | (ev.tag << 16);  // node_set_eval
        w->bits = ev.bits;
        w->std_dev = 0.0f;
    }
    Propagated p;
    if (ev_known(ev)) {
        p.eval = ev;
        p.variance = fmul(std_dev, std_dev);
    } else {
        const float negated = ev_notnan(ev_negate(child.eval));
        const float n = (float)t.visits[slot];
        float m = __uint_as_float(ev.bits);
        m = fadd(m, fdiv(fadd(fneg(m), negated), n));
        std_dev = fadd(std_dev, fdiv(fadd(fneg(std_dev), fsqrt(child.variance)), n));
        w->kind = 2;
        w->bits = __float_as_uint(m);
        w->std_dev = std_dev;
        p.eval = ev_value(fmul(negated, 0.997f));
        p.variance = fmul(fmul(child.variance, 0.997f), 0.997f);
    }
    return p;
}

__device__ __forceinline__ void warp_propagate_store(const GameTree& t, const PendingNode& w, int lane) {
    if (lane == 0 && w.kind != 0) {
        if (w.kind == 1) t.meta[w.slot] = w.meta;
        t.eval[w.slot] = w.bits;
        t.std_dev[w.slot] = w.std_dev;
    }
    __syncwarp();
}

// unwind `p` from the parent of the leaf (traj[len-2]) to the simulation root (traj[0])
__device__ __forceinline__ void warp_backup(const GameTree& t, const uint32_t* traj, int len,
                                            Propagated p, int lane) {
    for (int d = len - 2; d >= 0; d--) p = warp_propagate(t, traj[d], p, lane);
}
