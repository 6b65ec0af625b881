// GPU-resident lock-step PV-MCTS (reference pv_mcts.py:20-95).  G independent games each own a node
// arena; every simulation is three steps shared by all games:
//   aq_mcts_select         descend from the root with PUCT (pv_mcts.py:69-78) to a leaf, rebuilding
//                          the leaf's state by applying the actions on the path (lazy State.next)
//   (leaf evaluation)      aq_leaf_eval on the G leaf states = batched model.predict (pv_mcts.py:47)
//   aq_mcts_expand_backup  create the children in legal_actions() order with their priors
//                          (pv_mcts.py:53-56) and back the value up with alternating sign (:60-66)
// The reference has no virtual loss, no Dirichlet noise and no tree reuse, so batching ACROSS games
// leaves every game's search unchanged.  Tree reuse between moves (aq_mcts_advance, AlphaGo Zero) and
// Dirichlet noise on the root priors (aq_mcts_root_noise, AlphaZero) are opt-in additions the reference
// does not have; without them every search starts from aq_mcts_reset with the network's priors.
//
// Arithmetic is kept as the reference computes it under NumPy >= 2 (requirements.txt pins
// numpy~=2.0.2, NEP 50 promotion): w accumulates in float64; the PUCT score is
//   float32(-w/n computed in float64) + ((float32(1.25) * p) * float32(sqrt(t))) / float32(1 + n)
// all in float32, and np.argmax takes the FIRST maximum.
#include <cfloat>

#include "aq_common.cuh"

using namespace aq;

// A node is split into the 16 bytes the PUCT scan of a parent reads for EVERY child (w, prior, n) and the 16 bytes only the chosen
// child needs (links, action): the selection kernel is bound by the bytes of the children it scans (133 children per level).
struct __align__(16) MctsHot {
    double w;           // cumulative value
    float prior;        // p
    int n;              // visit count
};
struct __align__(16) MctsCold {
    int first_child;    // -1 = not expanded
    int parent;         // -1 = root
    short n_children;
    short action;       // action that leads here from the parent
    int pad;            // 0; a child of a Gumbel root: the bits of its float base score (aq_mcts_gumbel_root)
};
static_assert(sizeof(MctsHot) == 16 && sizeof(MctsCold) == 16, "node halves must be 16 bytes");
constexpr size_t kNodeBytes = sizeof(MctsHot) + sizeof(MctsCold);

struct __align__(16) MctsGame {
    AqState root;
    int node_count;
    int leaf;       // node selected by the last aq_mcts_select
    int leaf_kind;  // 0 = evaluate with the network, 1 = terminal loss (-1), 2 = terminal draw (0)
    int overflow;   // arena exhausted (caller error: max_nodes too small)
    int pad[4];     // pad[0] != 0: the root's priors carry Dirichlet noise (aq_mcts_root_noise); reset / advance zero it
                    // pad[1..3]: the Gumbel root (aq_mcts_gumbel_root): the bits of v_hat (float), m (0 = no Gumbel root), n
};
static_assert(sizeof(MctsGame) == 64, "MctsGame must be 64 bytes");

static inline size_t mcts_nodes_offset(int64_t G) { return ((size_t)G * sizeof(MctsGame) + 255) & ~(size_t)255; }

// root node: Node(state, 0), pv_mcts.py:81
__device__ __forceinline__ void write_fresh_root(MctsHot *hot, MctsCold *cold) {
    MctsHot rh;
    rh.w = 0.0; rh.prior = 0.f; rh.n = 0;
    MctsCold rc;
    rc.first_child = -1; rc.parent = -1; rc.n_children = 0; rc.action = -1; rc.pad = 0;
    hot[0] = rh;
    cold[0] = rc;
}

// A game at the start of a search: nothing selected, no overflow, root priors without noise.
__device__ __forceinline__ MctsGame start_game(const AqState &root, int node_count) {
    MctsGame gm = {};
    gm.root = root;
    gm.node_count = node_count;
    return gm;
}

__global__ void mcts_reset_kernel(MctsGame *games, MctsHot *hot, MctsCold *cold, const AqState *__restrict__ roots, int64_t G,
                                  int64_t max_nodes) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    games[g] = start_game(load_state(roots + g), 1);
    write_fresh_root(hot + g * max_nodes, cold + g * max_nodes);
}

__device__ __forceinline__ bool same_position(const AqState &a, const AqState &b) {
    return a.hwalls == b.hwalls && a.vwalls == b.vwalls && a.ppos == b.ppos && a.pwalls == b.pwalls && a.epos == b.epos &&
           a.ewalls == b.ewalls && a.plies == b.plies;
}

// Breadth-first copy of the subtree below source node `from` into a destination arena, the arena itself serving as the queue:
// node 0 is `from` (now a root), and every expanded node copied appends its children block at the tail, so blocks stay contiguous
// and in legal_actions() order.  A copied node's first_child still holds the SOURCE index until the node is dequeued; the dequeue
// appends that block and rewrites it.  Returns the node count, or 0 when tail + reserve_nodes would pass max_nodes: the copy
// stops there and the caller writes a fresh root, so nothing depends on how far it had got.
__device__ int copy_subtree(const MctsHot *__restrict__ shot, const MctsCold *__restrict__ scold, int from, MctsHot *hot, MctsCold *cold,
                            int lane, int64_t max_nodes, int64_t reserve_nodes) {
    if (lane == 0) {
        hot[0] = shot[from];
        MctsCold rc = scold[from];
        rc.parent = -1;
        rc.action = -1;
        cold[0] = rc;
    }
    int tail = 1;
    for (int head = 0; head < tail;) {
        __syncwarp();  // the window's records were written by other lanes of this warp
        const int end = min(head + 32, tail);
        int sfc = -1, snc = 0;
        if (head + lane < end) {
            const MctsCold c = cold[head + lane];
            sfc = c.first_child;
            snc = c.n_children;
        }
        unsigned expanded = __ballot_sync(0xffffffffu, sfc >= 0);
        while (expanded) {
            const int j = __ffs(expanded) - 1;
            expanded &= expanded - 1;
            const int fc = __shfl_sync(0xffffffffu, sfc, j), nc = __shfl_sync(0xffffffffu, snc, j);
            if ((int64_t)tail + nc + reserve_nodes > max_nodes) return 0;
            for (int c = lane; c < nc; c += 32) {
                hot[tail + c] = shot[fc + c];
                MctsCold cc = scold[fc + c];
                cc.parent = head + j;
                cold[tail + c] = cc;
            }
            if (lane == j) cold[head + j].first_child = tail;
            tail += nc;
        }
        head = end;
    }
    return tail;
}

// One warp per destination game (aq_mcts_advance): follow the path from the source game's root with a ballot over each children
// block, check the position reached against roots[g], then carry the subtree or start from a fresh root.
__global__ void __launch_bounds__(128)
mcts_advance_kernel(const MctsGame *__restrict__ src_games, const MctsHot *__restrict__ src_hot_all, const MctsCold *__restrict__ src_cold_all,
                    int64_t G_src, MctsGame *dst_games, MctsHot *dst_hot_all, MctsCold *dst_cold_all, int64_t G_dst, int64_t max_nodes,
                    const AqState *__restrict__ roots, const int64_t *__restrict__ src_game, const int16_t *__restrict__ path, int path_len,
                    int64_t reserve_nodes, int32_t *__restrict__ kept, int32_t *__restrict__ status) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G_dst) return;
    MctsHot *hot = dst_hot_all + g * max_nodes;
    MctsCold *cold = dst_cold_all + g * max_nodes;
    const AqState root = load_state(roots + g);
    const int64_t s = src_game[g];
    int count = 0;  // nodes carried, 0 = fresh root
    if (s < -1 || s >= G_src) {
        if (lane == 0) atomicAdd(status, 1);
    } else if (s >= 0) {
        const MctsHot *shot = src_hot_all + s * max_nodes;
        const MctsCold *scold = src_cold_all + s * max_nodes;
        AqState st = load_state(&src_games[s].root);
        int node = 0;  // -1 once the path leaves the tree
        for (int i = 0; i < path_len; ++i) {
            const int a = path[g * path_len + i];
            st = state_after(st, a);
            if (node < 0) continue;
            const int first = scold[node].first_child, nc = first < 0 ? 0 : scold[node].n_children;
            int found = -1;
            for (int c0 = 0; c0 < nc && found < 0; c0 += 32) {
                const int c = c0 + lane;
                const unsigned hit = __ballot_sync(0xffffffffu, c < nc && scold[first + c].action == a);
                if (hit) found = first + c0 + __ffs(hit) - 1;
            }
            node = found;
        }
        if (!same_position(st, root)) {
            if (lane == 0) atomicAdd(status, 1);
        } else if (node >= 0 && shot[node].n >= 1) {
            count = copy_subtree(shot, scold, node, hot, cold, lane, max_nodes, reserve_nodes);
        }
    }
    __syncwarp();
    if (lane == 0) {
        if (count == 0) write_fresh_root(hot, cold);
        dst_games[g] = start_game(root, count ? count : 1);
        if (kept) kept[g] = count;
    }
}

// ------------------------------------------------------------------------------------------
// Gumbel root (Gumbel AlphaZero: Danihelka et al., ICLR 2022; DeepMind mctx gumbel_muzero_policy; the reference has none).  Every
// node below the root keeps PUCT.  For a game whose root has K children with priors p_c (legal_actions() order) and
// logit_c = log p_c (-inf for p_c = 0), aq_mcts_gumbel_root stores, once, right after simulation 1 expanded the root (root.n == 1):
//   g_c    = gumbel_scale * (-log(-log U_c)),  U_c a splitmix64 counter draw keyed by (seed, game_id, ply) (mcts_gumbel_root_kernel)
//   base_c = float32(g_c + (logit_c - max logit))   in the root child's MctsCold.pad
//   v_hat  = root.w (the network value of the root), m = min(considered, K), n = sims - 1 (root-child visits of the search)
// At every root descent and in the result, with n_c, w_c the children's visits and values and N = sum n_c:
//   q_c    = -(w_c / n_c) for n_c > 0 (the root mover's view, as the PUCT scan reads it)
//   v_mix  = (v_hat + N * (S_pq / S_p)) / (N + 1),  S_p = sum_{n_c>0} pt_c, S_pq = sum_{n_c>0} pt_c * q_c, pt = max(p, FLT_MIN)
//            (S_pq / S_p taken as 0 when N = 0)
//   cq_c   = q_c if n_c > 0 else v_mix;  qh_c = (cq_c - min cq) / max(max cq - min cq, 1e-8)
//   sigma_c = ((50 + max_b n_b) * 0.1) * qh_c                                          (mctx maxvisit_init = 50, value_scale = 0.1)
//   score_c = max(-1e9, base_c + sigma_c)
//   descent at simulation index k = N: the first argmax of score_c over the children with n_c == considered_visit(m, n, k)
//   choice: the first argmax of score_c over the children with n_c == max_b n_b;  improved policy: softmax(logit_c + sigma_c)
// (no child matching: child 0, as jnp.argmax over all -inf).  Scores are float64 with every operation rounded as written; sums
// run in warp order: lane l adds its children l, l + 32, ... in order from 0.0, then S_l += S_(l xor m) for m = 16, 8, 4, 2, 1.
// tests/mcts_gumbel_oracle.py restates all of it.
// ------------------------------------------------------------------------------------------

// mctx get_sequence_of_considered_visits(m, n)[k] (sequential halving), continued past k = n - 1 by the same rule: phases of
// `extra` rounds over the first nc children, extra = max(1, n / (ceil(log2 m) * nc)), nc halving from m down to 2.  The children a
// phase considers have equal visit counts, so entry k of a phase is the visits before it plus k / nc.
__device__ __forceinline__ int considered_visit(int m, int n, int k) {
    if (m <= 1) return k;
    const int log2max = 32 - __clz(m - 1);
    int nc = m, base = 0;
    while (true) {
        const int extra = max(1, n / (log2max * nc));
        if (k < extra * nc) return base + k / nc;
        k -= extra * nc;
        base += extra;
        nc = max(2, nc / 2);
    }
}

struct GumbelQ {
    double v_mix, q_lo, q_range, visit_scale;
    int max_n;
};

__device__ __forceinline__ double completed_q(const MctsHot &ch, double v_mix) { return ch.n > 0 ? -__ddiv_rn(ch.w, (double)ch.n) : v_mix; }

__device__ __forceinline__ double warp_sum(double s) {
#pragma unroll
    for (int m = 16; m; m >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, m));
    return s;
}

// What completes and rescales the root children's Q values (N = sum of their visits); the same in every lane.
__device__ __forceinline__ GumbelQ gumbel_q(const MctsGame &gm, const MctsHot *hot, int first, int nc, int N, int lane) {
    double sp = 0.0, spq = 0.0;
    int mx = 0;
#pragma unroll 1
    for (int c = lane; c < nc; c += 32) {
        const MctsHot ch = hot[first + c];
        const double pt = ch.n > 0 ? (double)fmaxf(ch.prior, FLT_MIN) : 0.0;
        sp = __dadd_rn(sp, pt);
        spq = __dadd_rn(spq, ch.n > 0 ? __dmul_rn(pt, completed_q(ch, 0.0)) : 0.0);
        mx = max(mx, ch.n);
    }
    sp = warp_sum(sp);
    spq = warp_sum(spq);
    GumbelQ r;
    r.max_n = __reduce_max_sync(0xffffffffu, mx);
    const double v_hat = (double)__int_as_float(gm.pad[1]);
    r.v_mix = __ddiv_rn(__dadd_rn(v_hat, __dmul_rn((double)N, N > 0 ? __ddiv_rn(spq, sp) : 0.0)), (double)(N + 1));
    double lo = INFINITY, hi = -INFINITY;
#pragma unroll 1
    for (int c = lane; c < nc; c += 32) {
        const double q = completed_q(hot[first + c], r.v_mix);
        lo = fmin(lo, q);
        hi = fmax(hi, q);
    }
#pragma unroll
    for (int m = 16; m; m >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, m));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, m));
    }
    r.q_lo = lo;
    r.q_range = fmax(__dsub_rn(hi, lo), 1e-8);
    r.visit_scale = __dmul_rn(__dadd_rn(50.0, (double)r.max_n), 0.1);
    return r;
}

__device__ __forceinline__ double gumbel_sigma(const GumbelQ &r, const MctsHot &ch) {
    return __dmul_rn(r.visit_scale, __ddiv_rn(__dsub_rn(completed_q(ch, r.v_mix), r.q_lo), r.q_range));
}

// First argmax of score_c over the root children with n_c == visits (child 0 when there is none); the same in every lane.
__device__ __forceinline__ int gumbel_pick(const GumbelQ &r, const MctsHot *hot, const MctsCold *cold, int first, int nc, int visits, int lane) {
    double best = -INFINITY;
    int best_c = 0x7fffffff;
#pragma unroll 1
    for (int c = lane; c < nc; c += 32) {
        const MctsHot ch = hot[first + c];
        if (ch.n != visits) continue;
        const double sc = fmax(-1e9, __dadd_rn((double)__int_as_float(cold[first + c].pad), gumbel_sigma(r, ch)));
        if (sc > best || best_c == 0x7fffffff) { best = sc; best_c = c; }   // ascending c: the first maximum of the lane
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, d);
        const int oc = __shfl_xor_sync(0xffffffffu, best_c, d);
        const bool take = (oc != 0x7fffffff) && (best_c == 0x7fffffff || ob > best || (ob == best && oc < best_c));
        if (take) { best = ob; best_c = oc; }
    }
    return best_c == 0x7fffffff ? 0 : best_c;
}

// Descent of game g by its warp (pv_mcts.py:69-78).  The node arrays are read through plain pointers: in the fused kernel the same
// warp has just written them (expansion + backup), so the loads must be coherent ones.  kGumbel: the root of a game with a Gumbel
// root (MctsGame.pad[2] > 0) is left by the Gumbel rule, every other node by PUCT.
template <bool kGumbel>
__device__ __forceinline__ void select_game(MctsGame *games, const MctsHot *hot, const MctsCold *cold, int64_t g, int lane, float c_puct,
                                            AqState *leaf_states, int32_t *leaf_kind) {
    AqState s = games[g].root;
    int node = 0, kind = 0;
    // what the descent needs from a node: first_child, n_children (cold half) and n (hot half, known from the scan of its parent)
    int first = cold[0].first_child, nc = cold[0].n_children, nn = hot[0].n;
    if (kGumbel && games[g].pad[2] > 0 && first >= 0 && nc > 0 && !terminal_flags(s)) {   // the Gumbel root's step; PUCT below it
        const MctsGame &gm = games[g];
        const GumbelQ r = gumbel_q(gm, hot, first, nc, nn - 1, lane);
        node = first + gumbel_pick(r, hot, cold, first, nc, considered_visit(gm.pad[2], gm.pad[3], nn - 1), lane);
        nn = hot[node].n;
        const MctsCold cc = cold[node];
        first = cc.first_child;
        nc = cc.n_children;
        s = state_after(s, cc.action);
    }
    while (true) {
        const int tf = terminal_flags(s);  // pv_mcts.py:35-42: terminal test comes first
        if (tf) { kind = (tf & 1) ? 1 : 2; break; }
        if (first < 0 || nc <= 0) { kind = 0; break; }  // `not self.child_nodes` (None or empty)
        // t = sum(child.n) (pv_mcts.py:70-72) = n - 1: the visit that expanded this node went to no child, every later
        // visit went to exactly one (terminal children count their visits too)
        const int t = nn - 1;
        const float sq = (float)sqrt((double)t);
        float best = -INFINITY;
        int best_c = 0x7fffffff;
        int b_n = 0;  // visit count of this lane's best child
        for (int c = lane; c < nc; c += 32) {
            const MctsHot ch = hot[first + c];
            const float q = ch.n ? (float)(-ch.w / (double)ch.n) : 0.0f;
            const float u = __fdiv_rn(__fmul_rn(__fmul_rn(c_puct, ch.prior), sq), (float)(1 + ch.n));
            const float sc = __fadd_rn(q, u);
            if (sc > best || (sc == best && c < best_c) || best_c == 0x7fffffff) {
                best = sc; best_c = c;
                b_n = ch.n;
            }
        }
        // warp arg-max, lowest index among equal maxima (np.argmax)
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, d);
            const int oc = __shfl_xor_sync(0xffffffffu, best_c, d);
            const bool take = (oc != 0x7fffffff) && (best_c == 0x7fffffff || ob > best || (ob == best && oc < best_c));
            if (take) { best = ob; best_c = oc; }
        }
        const int owner = best_c & 31;  // child c is examined by lane c % 32, whose own best is then the global best
        node = first + best_c;
        nn = __shfl_sync(0xffffffffu, b_n, owner);
        const MctsCold cc = cold[node];  // one 16-byte record of the chosen child
        first = cc.first_child;
        nc = cc.n_children;
        s = state_after(s, cc.action);  // lazy State.next along the path
    }
    if (lane == 0) {
        games[g].leaf = node;
        games[g].leaf_kind = kind;
        store_state(leaf_states + g, s);
        leaf_kind[g] = kind;
    }
}

// one warp per game
__global__ void __launch_bounds__(128)
mcts_select_kernel(MctsGame *games, const MctsHot *hot_all, const MctsCold *cold_all, int64_t G, int64_t max_nodes, float c_puct,
                   AqState *leaf_states, int32_t *leaf_kind) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    select_game<false>(games, hot_all + g * max_nodes, cold_all + g * max_nodes, g, lane, c_puct, leaf_states, leaf_kind);
}

// mcts_select_kernel with the Gumbel rule at the roots of games that have one
__global__ void __launch_bounds__(128)
mcts_select_gumbel_kernel(MctsGame *games, const MctsHot *hot_all, const MctsCold *cold_all, int64_t G, int64_t max_nodes, float c_puct,
                          AqState *leaf_states, int32_t *leaf_kind) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    select_game<true>(games, hot_all + g * max_nodes, cold_all + g * max_nodes, g, lane, c_puct, leaf_states, leaf_kind);
}

// Expansion of the selected leaf of game g with the evaluated priors (pv_mcts.py:47-56) and the backup of its value (:60-66).
__device__ __forceinline__ void expand_backup_game(MctsGame *games, MctsHot *hot, MctsCold *cold, int64_t g, int lane, int64_t max_nodes,
                                                   const float *priors, const float *values, const uint32_t *mask, const uint8_t *pawn) {
    const int leaf = games[g].leaf, kind = games[g].leaf_kind;
    double value;
    if (kind == 0) {
        value = (double)values[g];  // value.item(): float32 -> python float
        // children in State.legal_actions() order: ordered pawn moves, then per slot H before V
        const uint32_t *m = mask + 8 * g;
        const float *pr = priors + (int64_t)AQ_ACTIONS * g;
        const int np = pawn[8 * g];
        const int first = games[g].node_count;
        int total = np;
        // wall actions = mask bits >= 81 (word 2 holds actions 64..95); counted first to bound-check the arena
        int wl = 0;
        if (lane >= 2 && lane < 8) {
            uint32_t w = m[lane];
            if (lane == 2) w >>= 17;
            wl = __popc(w);
        }
        wl = __reduce_add_sync(0xffffffffu, wl);
        total += wl;
        bool fits = (int64_t)first + total <= max_nodes;
        if (!fits) {
            if (lane == 0) games[g].overflow = 1;
            total = 0;
        }
        if (fits) {
            MctsHot ch;
            ch.w = 0.0; ch.n = 0;
            MctsCold cc;
            cc.first_child = -1; cc.parent = leaf; cc.n_children = 0; cc.pad = 0;
            if (lane < np) {
                const int a = pawn[8 * g + 1 + lane];
                cc.action = (short)a;
                ch.prior = pr[a];
                hot[first + lane] = ch;
                cold[first + lane] = cc;
            }
            int base = first + np;
            for (int k = 0; k < 4; ++k) {
                const int c = lane + 32 * k;  // interleaved candidate index: 2*slot + (0 = H, 1 = V)
                const int slot = c >> 1;
                const int a = (c & 1) ? (AQ_SQUARES + AQ_SLOTS + slot) : (AQ_SQUARES + slot);
                const bool on = (m[a >> 5] >> (a & 31)) & 1;
                const unsigned bal = __ballot_sync(0xffffffffu, on);
                if (on) {
                    const int at = base + __popc(bal & ((1u << lane) - 1));
                    cc.action = (short)a;
                    ch.prior = pr[a];
                    hot[at] = ch;
                    cold[at] = cc;
                }
                base += __popc(bal);
            }
        }
        if (lane == 0) {
            cold[leaf].first_child = first;
            cold[leaf].n_children = (short)total;
            games[g].node_count = first + total;
        }
    } else {
        value = kind == 1 ? -1.0 : 0.0;  // pv_mcts.py:39
    }
    __syncwarp();
    if (lane == 0) {
        int node = leaf;
        while (node >= 0) {  // pv_mcts.py:50-51, 63-65: w += value; n += 1; parent gets -value
            hot[node].w += value;
            hot[node].n += 1;
            value = -value;
            node = cold[node].parent;
        }
    }
}

__global__ void __launch_bounds__(128)
mcts_expand_backup_kernel(MctsGame *games, MctsHot *hot_all, MctsCold *cold_all, int64_t G, int64_t max_nodes,
                          const float *__restrict__ priors, const float *__restrict__ values,
                          const uint32_t *__restrict__ mask, const uint8_t *__restrict__ pawn) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    expand_backup_game(games, hot_all + g * max_nodes, cold_all + g * max_nodes, g, lane, max_nodes, priors, values, mask, pawn);
}

// Expansion + backup of simulation i and the descent of simulation i + 1 in one launch: a game's next descent only needs that game's
// own backup, so there is no reason to wait for the other 4,095 games and for a kernel boundary in between.
__global__ void __launch_bounds__(128)
mcts_expand_select_kernel(MctsGame *games, MctsHot *hot_all, MctsCold *cold_all, int64_t G, int64_t max_nodes,
                          const float *__restrict__ priors, const float *__restrict__ values, const uint32_t *__restrict__ mask,
                          const uint8_t *__restrict__ pawn, float c_puct, AqState *leaf_states, int32_t *leaf_kind) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    MctsHot *hot = hot_all + g * max_nodes;
    MctsCold *cold = cold_all + g * max_nodes;
    expand_backup_game(games, hot, cold, g, lane, max_nodes, priors, values, mask, pawn);
    __syncwarp();   // orders the warp's node writes (children by all lanes, the backup by lane 0) before the descent's reads
    select_game<false>(games, hot, cold, g, lane, c_puct, leaf_states, leaf_kind);
}

// mcts_expand_select_kernel with the Gumbel rule at the roots of games that have one
__global__ void __launch_bounds__(128)
mcts_expand_select_gumbel_kernel(MctsGame *games, MctsHot *hot_all, MctsCold *cold_all, int64_t G, int64_t max_nodes,
                                 const float *__restrict__ priors, const float *__restrict__ values, const uint32_t *__restrict__ mask,
                                 const uint8_t *__restrict__ pawn, float c_puct, AqState *leaf_states, int32_t *leaf_kind) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    MctsHot *hot = hot_all + g * max_nodes;
    MctsCold *cold = cold_all + g * max_nodes;
    expand_backup_game(games, hot, cold, g, lane, max_nodes, priors, values, mask, pawn);
    __syncwarp();
    select_game<true>(games, hot, cold, g, lane, c_puct, leaf_states, leaf_kind);
}

__global__ void mcts_root_counts_kernel(const MctsGame *__restrict__ games, const MctsHot *__restrict__ hot_all,
                                        const MctsCold *__restrict__ cold_all, int64_t G, int64_t max_nodes, int32_t *__restrict__ counts,
                                        int16_t *__restrict__ actions, int16_t *__restrict__ n_out,
                                        int32_t *__restrict__ overflow) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    const MctsHot *hot = hot_all + g * max_nodes;
    const MctsCold *cold = cold_all + g * max_nodes;
    const int first = cold[0].first_child;
    const int nc = first < 0 ? 0 : cold[0].n_children;
    for (int c = lane; c < AQ_MAX_LEGAL; c += 32) {
        counts[g * AQ_MAX_LEGAL + c] = c < nc ? hot[first + c].n : 0;
        actions[g * AQ_MAX_LEGAL + c] = c < nc ? cold[first + c].action : (int16_t)-1;
    }
    if (lane == 0) {
        n_out[g] = (int16_t)nc;
        if (overflow && games[g].overflow) atomicExch(overflow, 1);
    }
}

// One warp per game, child c in lane c % 32 (as mcts_root_counts_kernel), every value in double as written:
//   root_value = w_root / n_root (the root mover's view; NaN if n_root == 0)
//   best_child = the child with the largest n, the first in legal_actions() order on ties (policy_from_counts(counts, 0)); -1 if none
//   best_q     = -(w_b / n_b) (the root mover's view); -inf if there is no child or n_b == 0
__global__ void __launch_bounds__(128)
mcts_root_values_kernel(const MctsHot *__restrict__ hot_all, const MctsCold *__restrict__ cold_all, int64_t G, int64_t max_nodes,
                        double *__restrict__ root_value, double *__restrict__ best_q, int16_t *__restrict__ best_child) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    const MctsHot *hot = hot_all + g * max_nodes;
    const MctsCold *cold = cold_all + g * max_nodes;
    const int first = cold[0].first_child;
    const int nc = first < 0 ? 0 : cold[0].n_children;
    long long best = -1;
    for (int c = lane; c < nc; c += 32) best = max(best, ((long long)hot[first + c].n << 8) | (long long)(255 - c));   // largest n, then smallest c
#pragma unroll
    for (int d = 16; d; d >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, d));
    if (lane == 0) {
        const MctsHot r = hot[0];
        root_value[g] = r.n > 0 ? __ddiv_rn(r.w, (double)r.n) : (double)NAN;
        const int b = best < 0 ? -1 : 255 - (int)(best & 255);
        double q = -INFINITY;
        if (b >= 0) {
            const MctsHot ch = hot[first + b];
            if (ch.n > 0) q = -__ddiv_rn(ch.w, (double)ch.n);
        }
        best_q[g] = q;
        best_child[g] = (int16_t)b;
    }
}

// ------------------------------------------------------------------------------------------
// One ply of G lock-step self-play games after their searches (reference self_play.py:47-60): for every game
//   scores = counts ** (1 / temperature) / sum  (pv_mcts.py:88-95; temperature 0 = one-hot on the FIRST maximum, np.argmax)
//   policy[action] = score for the legal actions, 0 elsewhere, over all 209 actions  (self_play.py:51-54)
//   action = one draw from `scores` (self_play.py:57, np.random.choice(legal_actions, p=scores)): inverse CDF in
//            legal_actions() order of a counter-based uniform -- a hash of (seed, game id, ply), so a game's moves do not
//            depend on which other games are still running
//   state  = state.next(action) (self_play.py:60), with its terminal flags.
// One warp per game; child c of the root lives in lane c % 32, slot c / 32.
// kChosen (aq_selfplay_advance_chosen): policy[action] = child_policy[c] and the move is child choice[g], both from the search
// (the Gumbel root's improved policy and choice); no counts, temperature or draw.
// ------------------------------------------------------------------------------------------
constexpr int kChildSlots = (AQ_MAX_LEGAL + 31) / 32;

__device__ __forceinline__ uint64_t mix64(uint64_t z) {  // splitmix64 finaliser
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// kResign (aq_selfplay_advance_resign): s = max(root_value[g], best_q[g]) (NaN if either is); resign_min[game_id, ply & 1] takes
// min(., s) for every game (a NaN s leaves it); a game that is not a calibration game (resign_draw(seed, game_id) < calibration)
// and has s < v_resign resigns: its policy row is written as ever, no move is played and its term flags are 1 | 4.
// is_calibration[game_id] records the calibration bit the kernel used, so callers need not restate the draw.
constexpr uint64_t kResignDomain = 0xA4093822299F31D0ull;   // the fractional digits of pi after kGumbelDomain's

// u in [0, 1) of game `id`: the same for every ply of the game, so a game is a calibration game for its whole length
__device__ __forceinline__ double resign_draw(uint64_t seed, int64_t id) {
    return (double)(mix64(mix64((seed ^ kResignDomain) + 0x9E3779B97F4A7C15ull * (uint64_t)(id + 1))) >> 11) * 0x1p-53;
}

// The move kernels share this body; selfplay_move_kernel<T, kChosen> instantiates it without kResign, so its code is what it was
// before resignation existed.  tid is the kernel's threadIdx.x: read there, the compiler knows its range from __launch_bounds__.
template <typename T, bool kChosen, bool kResign>
__device__ __forceinline__ void
selfplay_move(unsigned tid, const AqState *__restrict__ states, const int32_t *__restrict__ counts, const int16_t *__restrict__ actions,
              const int16_t *__restrict__ n_children, const int64_t *__restrict__ game_id, int64_t G, double inv_t, int greedy,
              uint64_t seed, int ply, const float *__restrict__ child_policy, const int16_t *__restrict__ choice,
              T *__restrict__ policy, int16_t *__restrict__ chosen, AqState *__restrict__ moved, uint8_t *__restrict__ term,
              const double *__restrict__ root_value, const double *__restrict__ best_q, double v_resign, double calibration,
              double *__restrict__ resign_min, uint8_t *__restrict__ is_calibration) {
    __shared__ T rows[4][AQ_ACTIONS];
    const int lane = tid & 31, w = tid >> 5;
    const int64_t g = (int64_t)blockIdx.x * 4 + w;
    if (g >= G) return;
    const int n = n_children[g];
    double x[kChildSlots];
    int act[kChildSlots];
    int pick = -1;
    double total = 1.0;   // kChosen: child_policy is recorded as it is
    if constexpr (kChosen) {
#pragma unroll
        for (int k = 0; k < kChildSlots; ++k) {
            const int c = lane + 32 * k;
            act[k] = c < n ? (int)actions[g * AQ_MAX_LEGAL + c] : -1;
            x[k] = c < n ? (double)child_policy[g * AQ_MAX_LEGAL + c] : 0.0;
        }
        pick = choice[g];
        if (pick >= n) pick = -1;
    } else {
        long long best = -1;
#pragma unroll
        for (int k = 0; k < kChildSlots; ++k) {
            const int c = lane + 32 * k;
            const int cnt = c < n ? counts[g * AQ_MAX_LEGAL + c] : 0;
            act[k] = c < n ? (int)actions[g * AQ_MAX_LEGAL + c] : -1;
            x[k] = inv_t == 1.0 ? (double)cnt : (cnt > 0 ? pow((double)cnt, inv_t) : 0.0);
            if (c < n) best = max(best, ((long long)cnt << 8) | (long long)(255 - c));   // largest count, then smallest index
        }
        if (greedy) {
#pragma unroll
            for (int d = 16; d; d >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, d));
            const int arg = 255 - (int)(best & 255);
#pragma unroll
            for (int k = 0; k < kChildSlots; ++k) x[k] = (lane + 32 * k == arg && n > 0) ? 1.0 : 0.0;
        }
        // running sums in child order: a warp scan per slot on top of the slots before it (fixed order: deterministic)
        double cum[kChildSlots], base = 0.0;
#pragma unroll
        for (int k = 0; k < kChildSlots; ++k) {
            double v = x[k];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double up = __shfl_up_sync(0xffffffffu, v, d);
                if (lane >= d) v += up;
            }
            cum[k] = base + v;
            base = __shfl_sync(0xffffffffu, cum[k], 31);
        }
        total = base;
        const uint64_t bits = mix64(mix64(seed + 0x9E3779B97F4A7C15ull * (uint64_t)(game_id[g] + 1)) + 0xD1B54A32D192ED03ull * (uint64_t)(ply + 1));
        const double target = (double)(bits >> 11) * (1.0 / 9007199254740992.0) * total;   // u in [0, 1) times the sum
        int last = -1;
#pragma unroll
        for (int k = 0; k < kChildSlots; ++k) {
            const unsigned over = __ballot_sync(0xffffffffu, x[k] > 0.0 && target < cum[k]);
            const unsigned any = __ballot_sync(0xffffffffu, x[k] > 0.0);
            if (pick < 0 && over) pick = 32 * k + __ffs(over) - 1;
            if (any) last = 32 * k + 31 - __clz(any);
        }
        if (pick < 0) pick = last;   // target == total after rounding: the last child with a positive score
    }
    int a = -1;
#pragma unroll
    for (int k = 0; k < kChildSlots; ++k) {
        const int v = __shfl_sync(0xffffffffu, act[k], pick & 31);
        if ((pick >> 5) == k) a = v;
    }
    // dense policy row, staged so that the global stores are consecutive
    T *row = rows[w];
    for (int i = lane; i < AQ_ACTIONS; i += 32) row[i] = (T)0;
    __syncwarp();
#pragma unroll
    for (int k = 0; k < kChildSlots; ++k)
        if (act[k] >= 0) row[act[k]] = (T)(total > 0.0 ? x[k] / total : 0.0);   // x / sum(xs), pv_mcts.py:94
    __syncwarp();
    for (int i = lane; i < AQ_ACTIONS; i += 32) policy[g * AQ_ACTIONS + i] = row[i];
    if (lane == 0) {
        AqState t = load_state(states + g);
        int flags = 2;   // a root without children cannot move: reported as a draw (does not happen for non-terminal roots)
        bool resigned = false;
        if constexpr (kResign) {
            const int64_t id = game_id[g];
            const double rv = root_value[g], bq = best_q[g];
            const double s = (isnan(rv) || isnan(bq)) ? (double)NAN : fmax(rv, bq);
            double *m = resign_min + 2 * id + (ply & 1);
            *m = fmin(*m, s);
            const bool cal = resign_draw(seed, id) < calibration;
            is_calibration[id] = (uint8_t)cal;
            resigned = !cal && s < v_resign;
        }
        if (resigned) {
            flags = 1 | 4;
            a = -1;
        } else if (pick >= 0) {
            t = state_after(t, a);
            flags = terminal_flags(t);
        }
        store_state(moved + g, t);
        term[g] = (uint8_t)flags;
        if (chosen) chosen[g] = (int16_t)a;
    }
}

template <typename T, bool kChosen>
__global__ void __launch_bounds__(128)
selfplay_move_kernel(const AqState *__restrict__ states, const int32_t *__restrict__ counts, const int16_t *__restrict__ actions,
                     const int16_t *__restrict__ n_children, const int64_t *__restrict__ game_id, int64_t G, double inv_t, int greedy,
                     uint64_t seed, int ply, const float *__restrict__ child_policy, const int16_t *__restrict__ choice,
                     T *__restrict__ policy, int16_t *__restrict__ chosen, AqState *__restrict__ moved, uint8_t *__restrict__ term) {
    selfplay_move<T, kChosen, false>(threadIdx.x, states, counts, actions, n_children, game_id, G, inv_t, greedy, seed, ply, child_policy, choice, policy,
                                     chosen, moved, term, nullptr, nullptr, 0.0, 0.0, nullptr, nullptr);
}

template <typename T, bool kChosen>
__global__ void __launch_bounds__(128)
selfplay_move_resign_kernel(const AqState *__restrict__ states, const int32_t *__restrict__ counts, const int16_t *__restrict__ actions,
                            const int16_t *__restrict__ n_children, const int64_t *__restrict__ game_id, int64_t G, double inv_t, int greedy,
                            uint64_t seed, int ply, const float *__restrict__ child_policy, const int16_t *__restrict__ choice,
                            T *__restrict__ policy, int16_t *__restrict__ chosen, AqState *__restrict__ moved, uint8_t *__restrict__ term,
                            const double *__restrict__ root_value, const double *__restrict__ best_q, double v_resign, double calibration,
                            double *__restrict__ resign_min, uint8_t *__restrict__ is_calibration) {
    selfplay_move<T, kChosen, true>(threadIdx.x, states, counts, actions, n_children, game_id, G, inv_t, greedy, seed, ply, child_policy, choice, policy,
                                    chosen, moved, term, root_value, best_q, v_resign, calibration, resign_min,
                                    is_calibration);
}

// Survivors keep their order (games that ended leave; self_play.py:45 `while not state.is_done()`); one CTA, a block scan per
// 1,024 games.  For a game that ended: final_flags[game] = terminal flags of its last state, final_plies[game] = its length
// (kResign: a resigned game, term bit 2, played `ply` moves).
template <bool kResign>
__device__ __forceinline__ void
selfplay_compact(const AqState *__restrict__ moved, const uint8_t *__restrict__ term, const int64_t *__restrict__ game_id,
                 int64_t G, int ply, AqState *__restrict__ next_states, int64_t *__restrict__ next_game_id,
                 uint8_t *__restrict__ final_flags, int64_t *__restrict__ final_plies, int32_t *__restrict__ alive_count) {
    __shared__ int warp_total[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int base = 0;
    for (int64_t start = 0; start < G; start += 1024) {
        const int64_t i = start + threadIdx.x;
        const int flags = i < G ? (int)term[i] : 1;
        const bool alive = i < G && flags == 0;
        const unsigned m = __ballot_sync(0xffffffffu, alive);
        if (lane == 0) warp_total[w] = __popc(m);
        __syncthreads();
        int before = 0, all = 0;
        for (int v = 0; v < 32; ++v) {
            const int t = warp_total[v];
            before += v < w ? t : 0;
            all += t;
        }
        if (i < G) {
            const int64_t id = game_id[i];
            if (alive) {
                const int64_t o = base + before + __popc(m & ((1u << lane) - 1u));
                store_state(next_states + o, load_state(moved + i));
                next_game_id[o] = id;
            } else {
                final_flags[id] = (uint8_t)flags;
                final_plies[id] = (kResign && (flags & 4)) ? ply : ply + 1;
            }
        }
        base += all;
        __syncthreads();
    }
    if (threadIdx.x == 0) *alive_count = base;
}

__global__ void __launch_bounds__(1024)
selfplay_compact_kernel(const AqState *__restrict__ moved, const uint8_t *__restrict__ term, const int64_t *__restrict__ game_id,
                        int64_t G, int ply, AqState *__restrict__ next_states, int64_t *__restrict__ next_game_id,
                        uint8_t *__restrict__ final_flags, int64_t *__restrict__ final_plies, int32_t *__restrict__ alive_count) {
    selfplay_compact<false>(moved, term, game_id, G, ply, next_states, next_game_id, final_flags, final_plies, alive_count);
}

__global__ void __launch_bounds__(1024)
selfplay_compact_resign_kernel(const AqState *__restrict__ moved, const uint8_t *__restrict__ term, const int64_t *__restrict__ game_id,
                               int64_t G, int ply, AqState *__restrict__ next_states, int64_t *__restrict__ next_game_id,
                               uint8_t *__restrict__ final_flags, int64_t *__restrict__ final_plies, int32_t *__restrict__ alive_count) {
    selfplay_compact<true>(moved, term, game_id, G, ply, next_states, next_game_id, final_flags, final_plies, alive_count);
}

// ------------------------------------------------------------------------------------------
// Dirichlet noise on the root priors (AlphaZero; the reference has none).  For game g with K = n_children root children:
//   eta ~ Dirichlet(alpha, ..., alpha),  p'_c = float32((1 - fraction) * (double)p_c + fraction * eta_c)  (double, rounded once)
// eta is a pure function of (seed, game_id, ply, K, alpha).  Counter layout (tests/mcts_noise_oracle.py restates it):
//   key        = mix64(mix64((seed ^ kNoiseDomain) + 0x9E3779B97F4A7C15 * (game_id + 1)) + 0xD1B54A32D192ED03 * (ply + 1))
//                (the move draw of selfplay_move_kernel without the domain constant: the two draws are independent)
//   U(c, j)    = ((mix64(key + 0x9E3779B97F4A7C15 * (c * kNoiseDraws + j + 1)) >> 11) + 1) * 2^-53, in (0, 1]
//   gamma_c    : shape a = alpha + 1 if alpha < 1 else alpha, Marsaglia-Tsang with d = a - 1/3, k = 1 / sqrt(9 d).  Attempt
//                i = 0 .. kNoiseAttempts-1 takes x = sqrt(-2 log U(c,3i+1)) * cos(2 pi U(c,3i+2)) (Box-Muller), t = 1 + k x, and
//                accepts when t > 0 and log U(c,3i+3) < ((0.5 x x + d) - d v) + d log v with v = t t t: log G = log(d v).  No
//                attempt accepted (probability < 1e-20): log G = log d.  For alpha < 1: log gamma_c = log G + log U(c,0) / alpha.
//   eta_c      = exp(log gamma_c - max_k log gamma_k) / S, S summed as the warp does it: lane l adds its children l, l+32, ...
//                in order from 0.0, then S_l += S_(l xor m) for m = 16, 8, 4, 2, 1.
// The logs matter: at alpha = 0.03 U^(1/alpha) underflows to 0 for every child often enough to make the linear form 0/0.
// All double products and sums are rounded one at a time (no contraction), as numpy computes them.
// ------------------------------------------------------------------------------------------
constexpr uint64_t kNoiseDomain = 0x243F6A8885A308D3ull;   // fractional digits of pi
constexpr int kNoiseAttempts = 16;                          // Marsaglia-Tsang accepts > 95 % of attempts for a >= 1
constexpr int kNoiseDraws = 1 + 3 * kNoiseAttempts;         // counters per child: the boost uniform, then 3 per attempt

__device__ __forceinline__ double noise_uniform(uint64_t key, int c, int j) {
    const uint64_t bits = mix64(key + 0x9E3779B97F4A7C15ull * (uint64_t)(c * kNoiseDraws + j + 1));
    return (double)((bits >> 11) + 1) * 0x1p-53;
}

__device__ __forceinline__ double noise_log_gamma(uint64_t key, int c, double alpha) {
    const bool boost = alpha < 1.0;
    const double a = boost ? alpha + 1.0 : alpha;
    const double d = a - 1.0 / 3.0, k = 1.0 / sqrt(9.0 * d);
    double lg = log(d);
    for (int i = 0; i < kNoiseAttempts; ++i) {
        const double r = sqrt(-2.0 * log(noise_uniform(key, c, 3 * i + 1)));
        const double x = __dmul_rn(r, cos(__dmul_rn(6.283185307179586, noise_uniform(key, c, 3 * i + 2))));
        const double t = __dadd_rn(1.0, __dmul_rn(k, x));
        if (!(t > 0.0)) continue;
        const double v = __dmul_rn(__dmul_rn(t, t), t);
        const double rhs = __dadd_rn(__dsub_rn(__dadd_rn(__dmul_rn(__dmul_rn(0.5, x), x), d), __dmul_rn(d, v)), __dmul_rn(d, log(v)));
        if (log(noise_uniform(key, c, 3 * i + 3)) < rhs) {
            lg = log(__dmul_rn(d, v));
            break;
        }
    }
    if (boost) lg = __dadd_rn(lg, log(noise_uniform(key, c, 0)) / alpha);
    return lg;
}

// One warp per game, child c in lane c % 32 (as selfplay_move_kernel).  A root is noised when it is expanded and not yet noised.
__global__ void __launch_bounds__(128)
mcts_root_noise_kernel(MctsGame *games, MctsHot *hot_all, const MctsCold *__restrict__ cold_all, int64_t G, int64_t max_nodes,
                       const int64_t *__restrict__ game_id, uint64_t seed, int ply, double alpha, double fraction,
                       float *__restrict__ root_priors) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    MctsHot *hot = hot_all + g * max_nodes;
    const MctsCold *cold = cold_all + g * max_nodes;
    const int first = cold[0].first_child;
    const int nc = first < 0 ? 0 : cold[0].n_children;
    if (first >= 0 && games[g].pad[0] == 0) {
        const uint64_t id = game_id ? (uint64_t)game_id[g] : (uint64_t)g;
        const uint64_t key = mix64(mix64((seed ^ kNoiseDomain) + 0x9E3779B97F4A7C15ull * (id + 1)) + 0xD1B54A32D192ED03ull * (uint64_t)(ply + 1));
        double e[kChildSlots];
        double mx = -INFINITY;
#pragma unroll
        for (int s = 0; s < kChildSlots; ++s) {
            const int c = lane + 32 * s;
            e[s] = c < nc ? noise_log_gamma(key, c, alpha) : -INFINITY;
            mx = fmax(mx, e[s]);
        }
#pragma unroll
        for (int m = 16; m; m >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, m));
        double sum = 0.0;
#pragma unroll
        for (int s = 0; s < kChildSlots; ++s) {
            e[s] = lane + 32 * s < nc ? exp(e[s] - mx) : 0.0;
            sum = __dadd_rn(sum, e[s]);
        }
#pragma unroll
        for (int m = 16; m; m >>= 1) sum = __dadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, m));
        const double keep = 1.0 - fraction;
#pragma unroll
        for (int s = 0; s < kChildSlots; ++s) {
            const int c = lane + 32 * s;
            if (c < nc) {
                const double p = (double)hot[first + c].prior;
                hot[first + c].prior = (float)__dadd_rn(__dmul_rn(keep, p), __dmul_rn(fraction, e[s] / sum));
            }
        }
        if (lane == 0) games[g].pad[0] = 1;
    }
    if (root_priors) {
        __syncwarp();
        for (int c = lane; c < AQ_MAX_LEGAL; c += 32) root_priors[g * AQ_MAX_LEGAL + c] = c < nc ? hot[first + c].prior : 0.f;
    }
}

// ------------------------------------------------------------------------------------------
// Gumbel root state (the rule is stated above select_game).  The Gumbel draw of child c of game g:
//   key = mix64(mix64((seed ^ kGumbelDomain) + 0x9E3779B97F4A7C15 * (game_id + 1)) + 0xD1B54A32D192ED03 * (ply + 1))
//   U_c = ((mix64(key + 0x9E3779B97F4A7C15 * (c + 1)) >> 11) + 0.5) * 2^-53, in (0, 1)
// so a game's draw depends on (seed, game id, ply) alone, not on its batch, its row or padding rows.
// ------------------------------------------------------------------------------------------
constexpr uint64_t kGumbelDomain = 0x13198A2E03707344ull;   // the fractional digits of pi after kNoiseDomain's

// One warp per game, child c in lane c % 32.  A root gets its Gumbel state when simulation 1 has expanded it and nothing has
// visited it since (root.n == 1, so root.w is the network value) and it has none yet; any other root is left as it is.
__global__ void __launch_bounds__(128)
mcts_gumbel_root_kernel(MctsGame *games, const MctsHot *__restrict__ hot_all, MctsCold *cold_all, int64_t G, int64_t max_nodes,
                        const int64_t *__restrict__ game_id, uint64_t seed, int ply, int considered, double gumbel_scale, int sims,
                        float *__restrict__ root_scores) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    const MctsHot *hot = hot_all + g * max_nodes;
    MctsCold *cold = cold_all + g * max_nodes;
    const int first = cold[0].first_child;
    const int nc = first < 0 ? 0 : cold[0].n_children;
    if (nc > 0 && hot[0].n == 1 && games[g].pad[2] == 0) {
        const uint64_t id = game_id ? (uint64_t)game_id[g] : (uint64_t)g;
        const uint64_t key = mix64(mix64((seed ^ kGumbelDomain) + 0x9E3779B97F4A7C15ull * (id + 1)) + 0xD1B54A32D192ED03ull * (uint64_t)(ply + 1));
        double gd[kChildSlots], lg[kChildSlots];   // g_c, logit_c
        double mx = -INFINITY;
#pragma unroll
        for (int s = 0; s < kChildSlots; ++s) {
            const int c = lane + 32 * s;
            const double u = (double)((mix64(key + 0x9E3779B97F4A7C15ull * (uint64_t)(c + 1)) >> 11) + 0.5) * 0x1p-53;
            gd[s] = __dmul_rn(gumbel_scale, -log(-log(u)));
            lg[s] = c < nc ? log((double)hot[first + c].prior) : -INFINITY;
            mx = fmax(mx, lg[s]);
        }
#pragma unroll
        for (int m = 16; m; m >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, m));
#pragma unroll
        for (int s = 0; s < kChildSlots; ++s) {
            const int c = lane + 32 * s;
            if (c < nc) cold[first + c].pad = __float_as_int((float)__dadd_rn(gd[s], __dsub_rn(lg[s], mx)));
        }
        if (lane == 0) {
            games[g].pad[1] = __float_as_int((float)hot[0].w);
            games[g].pad[2] = min(considered, nc);
            games[g].pad[3] = sims - 1;
        }
    }
    if (root_scores) {
        __syncwarp();
        for (int c = lane; c < AQ_MAX_LEGAL; c += 32) root_scores[g * AQ_MAX_LEGAL + c] = c < nc ? __int_as_float(cold[first + c].pad) : 0.f;
    }
}

// One warp per game: the improved policy softmax(logit + sigma) over the root's children (0 beyond them) and the choice, the first
// argmax of the score over the most visited children.  A game without a Gumbel root: policy 0, choice -1.
__global__ void __launch_bounds__(128)
mcts_gumbel_result_kernel(const MctsGame *__restrict__ games, const MctsHot *__restrict__ hot_all, const MctsCold *__restrict__ cold_all,
                          int64_t G, int64_t max_nodes, float *__restrict__ policy, int16_t *__restrict__ choice) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= G) return;
    const MctsHot *hot = hot_all + g * max_nodes;
    const MctsCold *cold = cold_all + g * max_nodes;
    const MctsGame &gm = games[g];
    float *row = policy + g * AQ_MAX_LEGAL;
    if (gm.pad[2] <= 0) {
        for (int c = lane; c < AQ_MAX_LEGAL; c += 32) row[c] = 0.f;
        if (lane == 0) choice[g] = -1;
        return;
    }
    const int first = cold[0].first_child, nc = cold[0].n_children;
    const GumbelQ r = gumbel_q(gm, hot, first, nc, hot[0].n - 1, lane);
    const int pick = gumbel_pick(r, hot, cold, first, nc, r.max_n, lane);
    double z[kChildSlots];
    double mx = -INFINITY;
#pragma unroll
    for (int s = 0; s < kChildSlots; ++s) {
        const int c = lane + 32 * s;
        z[s] = -INFINITY;
        if (c < nc) {
            const MctsHot ch = hot[first + c];
            z[s] = __dadd_rn(log((double)ch.prior), gumbel_sigma(r, ch));
        }
        mx = fmax(mx, z[s]);
    }
#pragma unroll
    for (int m = 16; m; m >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, m));
    double sum = 0.0;
#pragma unroll
    for (int s = 0; s < kChildSlots; ++s) {
        z[s] = lane + 32 * s < nc ? exp(__dsub_rn(z[s], mx)) : 0.0;
        sum = __dadd_rn(sum, z[s]);
    }
    sum = warp_sum(sum);
#pragma unroll
    for (int s = 0; s < kChildSlots; ++s) {
        const int c = lane + 32 * s;
        if (c < AQ_MAX_LEGAL) row[c] = c < nc ? (float)__ddiv_rn(z[s], sum) : 0.f;
    }
    if (lane == 0) choice[g] = (int16_t)pick;
}

// ------------------------------------------------------------------------------------------
extern "C" int64_t aq_mcts_ws_bytes(int64_t G, int64_t max_nodes) {
    return (int64_t)(mcts_nodes_offset(G) + (size_t)G * (size_t)max_nodes * kNodeBytes);
}

static inline MctsGame *games_of(void *ws) { return reinterpret_cast<MctsGame *>(ws); }
// workspace: games | hot halves [G][max_nodes] | cold halves [G][max_nodes]
static inline MctsHot *hot_of(void *ws, int64_t G) {
    return reinterpret_cast<MctsHot *>(reinterpret_cast<unsigned char *>(ws) + mcts_nodes_offset(G));
}
static inline MctsCold *cold_of(void *ws, int64_t G, int64_t max_nodes) {
    return reinterpret_cast<MctsCold *>(reinterpret_cast<unsigned char *>(ws) + mcts_nodes_offset(G) + (size_t)G * (size_t)max_nodes * sizeof(MctsHot));
}

extern "C" int aq_mcts_reset(void *ws, const AqState *roots, int64_t G, int64_t max_nodes, void *stream) {
    if (G <= 0 || max_nodes < 1 || !ws || !roots) return aq_set_error(AQ_ERR_ARG, "aq_mcts_reset");
    return aq_launch("aq_mcts_reset", mcts_reset_kernel, (unsigned)((G + 127) / 128), 128, 0, reinterpret_cast<cudaStream_t>(stream), false,
                     games_of(ws), hot_of(ws, G), cold_of(ws, G, max_nodes), roots, G, max_nodes);
}

extern "C" int aq_mcts_advance(const void *src_ws, int64_t G_src, void *dst_ws, int64_t G_dst, int64_t max_nodes, const AqState *roots,
                               const int64_t *src_game, const int16_t *path, int path_len, int64_t reserve_nodes, int32_t *kept,
                               int32_t *status, void *stream) {
    if (G_src <= 0 || G_dst <= 0 || max_nodes < 1 || max_nodes > INT32_MAX || path_len < 1 || reserve_nodes < 0 ||
        reserve_nodes >= max_nodes || !src_ws || !dst_ws || !roots || !src_game || !path || !status)
        return aq_set_error(AQ_ERR_ARG, "aq_mcts_advance");
    const uintptr_t s0 = reinterpret_cast<uintptr_t>(src_ws), d0 = reinterpret_cast<uintptr_t>(dst_ws);
    const uintptr_t s1 = s0 + (uintptr_t)aq_mcts_ws_bytes(G_src, max_nodes), d1 = d0 + (uintptr_t)aq_mcts_ws_bytes(G_dst, max_nodes);
    if (s0 < d1 && d0 < s1) return aq_set_error(AQ_ERR_ARG, "aq_mcts_advance: the workspaces overlap");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(status, 0, sizeof(int32_t), st);
    if (e != cudaSuccess) return aq_set_error((int)e, "aq_mcts_advance");
    void *src = const_cast<void *>(src_ws);
    return aq_launch("aq_mcts_advance", mcts_advance_kernel, (unsigned)((G_dst + 3) / 4), 128, 0, st, false, games_of(src), hot_of(src, G_src),
                     cold_of(src, G_src, max_nodes), G_src, games_of(dst_ws), hot_of(dst_ws, G_dst), cold_of(dst_ws, G_dst, max_nodes), G_dst,
                     max_nodes, roots, src_game, path, path_len, reserve_nodes, kept, status);
}

extern "C" int aq_mcts_select(void *ws, int64_t G, int64_t max_nodes, float c_puct, AqState *leaf_states,
                              int32_t *leaf_kind, void *stream) {
    if (G <= 0 || !ws || !leaf_states || !leaf_kind) return aq_set_error(AQ_ERR_ARG, "aq_mcts_select");
    return aq_launch("aq_mcts_select", mcts_select_kernel, (unsigned)((G + 3) / 4), 128, 0, reinterpret_cast<cudaStream_t>(stream), false,
                     games_of(ws), hot_of(ws, G), cold_of(ws, G, max_nodes), G, max_nodes, c_puct, leaf_states, leaf_kind);
}

extern "C" int aq_mcts_select_gumbel(void *ws, int64_t G, int64_t max_nodes, float c_puct, AqState *leaf_states,
                                     int32_t *leaf_kind, void *stream) {
    if (G <= 0 || !ws || !leaf_states || !leaf_kind) return aq_set_error(AQ_ERR_ARG, "aq_mcts_select_gumbel");
    return aq_launch("aq_mcts_select_gumbel", mcts_select_gumbel_kernel, (unsigned)((G + 3) / 4), 128, 0, reinterpret_cast<cudaStream_t>(stream),
                     false, games_of(ws), hot_of(ws, G), cold_of(ws, G, max_nodes), G, max_nodes, c_puct, leaf_states, leaf_kind);
}

extern "C" int aq_mcts_expand_backup(void *ws, int64_t G, int64_t max_nodes, const float *priors, const float *values,
                                     const uint32_t *mask, const uint8_t *pawn, void *stream) {
    if (G <= 0 || !ws || !priors || !values || !mask || !pawn) return aq_set_error(AQ_ERR_ARG, "aq_mcts_expand_backup");
    return aq_launch("aq_mcts_expand_backup", mcts_expand_backup_kernel, (unsigned)((G + 3) / 4), 128, 0, reinterpret_cast<cudaStream_t>(stream),
                     false, games_of(ws), hot_of(ws, G), cold_of(ws, G, max_nodes), G, max_nodes, priors, values, mask, pawn);
}

extern "C" int aq_mcts_expand_select(void *ws, int64_t G, int64_t max_nodes, const float *priors, const float *values, const uint32_t *mask,
                                     const uint8_t *pawn, float c_puct, AqState *leaf_states, int32_t *leaf_kind, void *stream) {
    if (G <= 0 || !ws || !priors || !values || !mask || !pawn || !leaf_states || !leaf_kind) return aq_set_error(AQ_ERR_ARG, "aq_mcts_expand_select");
    return aq_launch("aq_mcts_expand_select", mcts_expand_select_kernel, (unsigned)((G + 3) / 4), 128, 0, reinterpret_cast<cudaStream_t>(stream),
                     false, games_of(ws), hot_of(ws, G), cold_of(ws, G, max_nodes), G, max_nodes, priors, values, mask, pawn, c_puct, leaf_states,
                     leaf_kind);
}

extern "C" int aq_mcts_expand_select_gumbel(void *ws, int64_t G, int64_t max_nodes, const float *priors, const float *values,
                                            const uint32_t *mask, const uint8_t *pawn, float c_puct, AqState *leaf_states, int32_t *leaf_kind,
                                            void *stream) {
    if (G <= 0 || !ws || !priors || !values || !mask || !pawn || !leaf_states || !leaf_kind)
        return aq_set_error(AQ_ERR_ARG, "aq_mcts_expand_select_gumbel");
    return aq_launch("aq_mcts_expand_select_gumbel", mcts_expand_select_gumbel_kernel, (unsigned)((G + 3) / 4), 128, 0,
                     reinterpret_cast<cudaStream_t>(stream), false, games_of(ws), hot_of(ws, G), cold_of(ws, G, max_nodes), G, max_nodes, priors,
                     values, mask, pawn, c_puct, leaf_states, leaf_kind);
}

extern "C" int aq_mcts_root_counts(void *ws, int64_t G, int64_t max_nodes, int32_t *counts, int16_t *actions,
                                   int16_t *n_children, int32_t *overflow, void *stream) {
    if (G <= 0 || !ws || !counts || !actions || !n_children) return aq_set_error(AQ_ERR_ARG, "aq_mcts_root_counts");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (overflow) {
        cudaError_t e = cudaMemsetAsync(overflow, 0, sizeof(int32_t), st);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_mcts_root_counts");
    }
    return aq_launch("aq_mcts_root_counts", mcts_root_counts_kernel, (unsigned)((G + 3) / 4), 128, 0, st, false, games_of(ws), hot_of(ws, G),
                     cold_of(ws, G, max_nodes), G, max_nodes, counts, actions, n_children, overflow);
}

extern "C" int aq_mcts_root_values(void *ws, int64_t G, int64_t max_nodes, double *root_value, double *best_q, int16_t *best_child,
                                   void *stream) {
    if (G <= 0 || max_nodes < 1 || !ws || !root_value || !best_q || !best_child) return aq_set_error(AQ_ERR_ARG, "aq_mcts_root_values");
    return aq_launch("aq_mcts_root_values", mcts_root_values_kernel, (unsigned)((G + 3) / 4), 128, 0, reinterpret_cast<cudaStream_t>(stream),
                     false, hot_of(ws, G), cold_of(ws, G, max_nodes), G, max_nodes, root_value, best_q, best_child);
}

extern "C" int aq_mcts_root_noise(void *ws, int64_t G, int64_t max_nodes, const int64_t *game_id, uint64_t seed, int32_t ply, float alpha,
                                  float fraction, float *root_priors, void *stream) {
    if (G < 1 || max_nodes < 1 || !ws || !(alpha > 0.f) || !isfinite(alpha) || !(fraction >= 0.f && fraction <= 1.f))
        return aq_set_error(AQ_ERR_ARG, "aq_mcts_root_noise");
    return aq_launch("aq_mcts_root_noise", mcts_root_noise_kernel, (unsigned)((G + 3) / 4), 128, 0, reinterpret_cast<cudaStream_t>(stream), false,
                     games_of(ws), hot_of(ws, G), cold_of(ws, G, max_nodes), G, max_nodes, game_id, seed, (int)ply, (double)alpha,
                     (double)fraction, root_priors);
}

extern "C" int aq_mcts_gumbel_root(void *ws, int64_t G, int64_t max_nodes, const int64_t *game_id, uint64_t seed, int32_t ply,
                                   int32_t considered, float gumbel_scale, int32_t sims, float *root_scores, void *stream) {
    if (G < 1 || max_nodes < 1 || !ws || considered < 1 || sims < 1 || !(gumbel_scale >= 0.f) || !isfinite(gumbel_scale))
        return aq_set_error(AQ_ERR_ARG, "aq_mcts_gumbel_root");
    return aq_launch("aq_mcts_gumbel_root", mcts_gumbel_root_kernel, (unsigned)((G + 3) / 4), 128, 0, reinterpret_cast<cudaStream_t>(stream), false,
                     games_of(ws), hot_of(ws, G), cold_of(ws, G, max_nodes), G, max_nodes, game_id, seed, (int)ply, (int)considered,
                     (double)gumbel_scale, (int)sims, root_scores);
}

extern "C" int aq_mcts_gumbel_result(void *ws, int64_t G, int64_t max_nodes, float *policy, int16_t *choice, void *stream) {
    if (G < 1 || max_nodes < 1 || !ws || !policy || !choice) return aq_set_error(AQ_ERR_ARG, "aq_mcts_gumbel_result");
    return aq_launch("aq_mcts_gumbel_result", mcts_gumbel_result_kernel, (unsigned)((G + 3) / 4), 128, 0, reinterpret_cast<cudaStream_t>(stream),
                     false, games_of(ws), hot_of(ws, G), cold_of(ws, G, max_nodes), G, max_nodes, policy, choice);
}

extern "C" int64_t aq_selfplay_ws_bytes(int64_t G) {
    return (int64_t)(((size_t)(G > 0 ? G : 0) * sizeof(AqState) + 255) & ~(size_t)255) + (G > 0 ? G : 0);
}

// What the resigning ply reads and writes besides the move (aq_selfplay_advance_resign).
struct ResignArgs {
    const double *root_value, *best_q;
    double v_resign, calibration;
    double *resign_min;
    uint8_t *is_calibration;
};

template <typename T, bool kChosen, bool kResign>
static int launch_move(const char *what, unsigned grid, cudaStream_t st, const AqState *states, const int32_t *counts, const int16_t *actions,
                       const int16_t *n_children, const int64_t *game_id, int64_t G, double inv_t, int greedy, uint64_t seed, int32_t ply,
                       const float *child_policy, const int16_t *choice, void *policy, int16_t *chosen, AqState *moved, uint8_t *term,
                       const ResignArgs &r) {
    if constexpr (kResign)
        return aq_launch(what, selfplay_move_resign_kernel<T, kChosen>, grid, 128, 0, st, false, states, counts, actions, n_children, game_id,
                         G, inv_t, greedy, seed, (int)ply, child_policy, choice, reinterpret_cast<T *>(policy), chosen, moved, term, r.root_value,
                         r.best_q, r.v_resign, r.calibration, r.resign_min, r.is_calibration);
    else
        return aq_launch(what, selfplay_move_kernel<T, kChosen>, grid, 128, 0, st, false, states, counts, actions, n_children, game_id, G,
                         inv_t, greedy, seed, (int)ply, child_policy, choice, reinterpret_cast<T *>(policy), chosen, moved, term);
}

// The move kernel of kChosen (and kResign), then the compaction of the games still running.
template <bool kChosen, bool kResign>
static int selfplay_advance(const char *what, const char *compact_what, const AqState *states, const int32_t *counts, const float *child_policy,
                            const int16_t *choice, const int16_t *actions, const int16_t *n_children, const int64_t *game_id, int64_t G,
                            double temperature, uint64_t seed, int32_t ply, void *policy, int policy_f64, int16_t *chosen, const ResignArgs &r,
                            AqState *next_states, int64_t *next_game_id, uint8_t *final_flags, int64_t *final_plies, int32_t *alive_count,
                            void *workspace, cudaStream_t st) {
    AqState *moved = reinterpret_cast<AqState *>(workspace);
    uint8_t *term = reinterpret_cast<uint8_t *>(workspace) + (((size_t)G * sizeof(AqState) + 255) & ~(size_t)255);
    const int greedy = temperature == 0.0;
    const double inv_t = greedy ? 1.0 : 1.0 / temperature;
    const unsigned grid = (unsigned)((G + 3) / 4);
    const int rc = (policy_f64 ? launch_move<double, kChosen, kResign> : launch_move<float, kChosen, kResign>)(
        what, grid, st, states, counts, actions, n_children, game_id, G, inv_t, greedy, seed, ply, child_policy, choice, policy, chosen, moved,
        term, r);
    if (rc) return rc;
    return aq_launch(compact_what, kResign ? selfplay_compact_resign_kernel : selfplay_compact_kernel, 1, 1024, 0, st, false, moved, term,
                     game_id, G, (int)ply, next_states, next_game_id, final_flags, final_plies, alive_count);
}

extern "C" int aq_selfplay_advance(const AqState *states, const int32_t *counts, const int16_t *actions, const int16_t *n_children,
                                   const int64_t *game_id, int64_t G, double temperature, uint64_t seed, int32_t ply, void *policy,
                                   int policy_f64, int16_t *chosen, AqState *next_states, int64_t *next_game_id, uint8_t *final_flags,
                                   int64_t *final_plies, int32_t *alive_count, void *workspace, void *stream) {
    if (G <= 0 || !states || !counts || !actions || !n_children || !game_id || !policy || !next_states || !next_game_id || !final_flags ||
        !final_plies || !alive_count || !workspace || !(temperature >= 0.0))
        return aq_set_error(AQ_ERR_ARG, "aq_selfplay_advance");
    return selfplay_advance<false, false>("aq_selfplay_advance(move)", "aq_selfplay_advance(compact)", states, counts, nullptr, nullptr,
                                          actions, n_children, game_id, G, temperature, seed, ply, policy, policy_f64, chosen, ResignArgs{},
                                          next_states, next_game_id, final_flags, final_plies, alive_count, workspace,
                                          reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int aq_selfplay_advance_chosen(const AqState *states, const float *child_policy, const int16_t *choice, const int16_t *actions,
                                          const int16_t *n_children, const int64_t *game_id, int64_t G, int32_t ply, void *policy,
                                          int policy_f64, int16_t *chosen, AqState *next_states, int64_t *next_game_id, uint8_t *final_flags,
                                          int64_t *final_plies, int32_t *alive_count, void *workspace, void *stream) {
    if (G <= 0 || !states || !child_policy || !choice || !actions || !n_children || !game_id || !policy || !next_states || !next_game_id ||
        !final_flags || !final_plies || !alive_count || !workspace)
        return aq_set_error(AQ_ERR_ARG, "aq_selfplay_advance_chosen");
    return selfplay_advance<true, false>("aq_selfplay_advance_chosen(move)", "aq_selfplay_advance_chosen(compact)", states, nullptr,
                                         child_policy, choice, actions, n_children, game_id, G, 1.0, 0, ply, policy, policy_f64, chosen,
                                         ResignArgs{}, next_states, next_game_id, final_flags, final_plies, alive_count, workspace,
                                         reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int aq_selfplay_advance_resign(const AqState *states, const int32_t *counts, const float *child_policy, const int16_t *choice,
                                          const int16_t *actions, const int16_t *n_children, const int64_t *game_id, int64_t G, double temperature,
                                          uint64_t seed, int32_t ply, void *policy, int policy_f64, int16_t *chosen, const double *root_value,
                                          const double *best_q, double v_resign, double calibration, double *resign_min, uint8_t *is_calibration,
                                          AqState *next_states,
                                          int64_t *next_game_id, uint8_t *final_flags, int64_t *final_plies, int32_t *alive_count, void *workspace,
                                          void *stream) {
    const bool by_counts = counts != nullptr, by_choice = child_policy != nullptr || choice != nullptr;
    if (G <= 0 || !states || by_counts == by_choice || (by_choice && (!child_policy || !choice)) || (by_counts && !(temperature >= 0.0)) ||
        !actions || !n_children || !game_id || !policy || !next_states || !next_game_id || !final_flags || !final_plies || !alive_count ||
        !workspace || isnan(v_resign) || !(calibration >= 0.0 && calibration <= 1.0) || !root_value || !best_q || !resign_min ||
        !is_calibration)
        return aq_set_error(AQ_ERR_ARG, "aq_selfplay_advance_resign");
    const ResignArgs r{root_value, best_q, v_resign, calibration, resign_min, is_calibration};
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (by_counts)
        return selfplay_advance<false, true>("aq_selfplay_advance_resign(move)", "aq_selfplay_advance_resign(compact)", states, counts, nullptr,
                                             nullptr, actions, n_children, game_id, G, temperature, seed, ply, policy, policy_f64, chosen, r,
                                             next_states, next_game_id, final_flags, final_plies, alive_count, workspace, st);
    return selfplay_advance<true, true>("aq_selfplay_advance_resign(move)", "aq_selfplay_advance_resign(compact)", states, nullptr, child_policy,
                                        choice, actions, n_children, game_id, G, 1.0, seed, ply, policy, policy_f64, chosen, r, next_states,
                                        next_game_id, final_flags, final_plies, alive_count, workspace, st);
}
