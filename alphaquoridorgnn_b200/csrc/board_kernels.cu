// Integer half of the hot path: game_logic.State on the GPU.
//   K1 legal_mask      game_logic.py:103-357
//   K2 build_graph     derived from game_logic.py:145-167 (edges) and 56-93 (features)
//   K9 state_next      game_logic.py:43-54, 359-391
// plus row68 <-> AqState packing and the ordered action list.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include "legal_steps.cuh"

// ------------------------------------------------------------------------------------------
// error plumbing (thread-local, no global mutable state shared between host threads)
// ------------------------------------------------------------------------------------------
static thread_local char g_err[256] = "ok";

int aq_set_error(int code, const char *what) {
    if (code > 0)
        snprintf(g_err, sizeof g_err, "%s: %s", what, cudaGetErrorString((cudaError_t)code));
    else
        snprintf(g_err, sizeof g_err, "%s: invalid argument", what);
    return code;
}

// every kernel launch of the library goes through aq_launch (aq_common.cuh), which ends in aq_check_launch: the successful ones are
// counted (aq_launch_count), so that a caller can state how many of this library's kernels ran in a region instead of assuming it
// (bench.py: gpu_launches)
static std::atomic<long long> g_launches{0};

int aq_check_launch(const char *what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return aq_set_error((int)e, what);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int64_t aq_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

int aq_num_sms() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0, n = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        sms = n > 0 ? n : 148;
    }
    return sms;
}

extern "C" int aq_version(void) { return AQ_VERSION; }
extern "C" const char *aq_last_error_string(void) { return g_err; }

using namespace aq;

// ------------------------------------------------------------------------------------------
// pack / unpack
// ------------------------------------------------------------------------------------------
__global__ void pack_states_kernel(const uint8_t *__restrict__ rows, const int16_t *__restrict__ plies, int64_t B,
                                   AqState *__restrict__ out) {
    // one warp per state: lanes 0..63 hold the wall entries (two per lane), ballot builds the bitboards
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const uint8_t *r = rows + 68 * b;
    const uint8_t w0 = r[4 + lane], w1 = r[4 + 32 + lane];
    const unsigned h0 = __ballot_sync(0xffffffffu, w0 == 1), h1 = __ballot_sync(0xffffffffu, w1 == 1);
    const unsigned v0 = __ballot_sync(0xffffffffu, w0 == 2), v1 = __ballot_sync(0xffffffffu, w1 == 2);
    if (lane == 0) {
        uint4 a;
        a.x = h0; a.y = h1; a.z = v0; a.w = v1;
        uint4 c;
        c.x = (unsigned)r[0] | ((unsigned)r[1] << 8) | ((unsigned)r[2] << 16) | ((unsigned)r[3] << 24);
        c.y = plies ? (unsigned)(uint16_t)plies[b] : 0u;
        c.z = 0; c.w = 0;
        uint4 *o = reinterpret_cast<uint4 *>(out + b);
        o[0] = a;
        o[1] = c;
    }
}

__global__ void unpack_states_kernel(const AqState *__restrict__ states, int64_t B, uint8_t *__restrict__ rows,
                                     int16_t *__restrict__ plies) {
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const AqState s = load_state(states + b);
    uint8_t *r = rows + 68 * b;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int slot = lane + 32 * k;
        r[4 + slot] = (uint8_t)(((s.hwalls >> slot) & 1) | (((s.vwalls >> slot) & 1) << 1));
    }
    if (lane == 0) {
        r[0] = s.ppos; r[1] = s.pwalls; r[2] = s.epos; r[3] = s.ewalls;
        if (plies) plies[b] = (int16_t)s.plies;
    }
}

// ------------------------------------------------------------------------------------------
// K1 legal_mask.  Three forms, all running the per-state steps of legal_steps.cuh: prepare (open-direction boards, can_place + gate of
// all 128 candidates, the witness paths of mover and opponent, and the (candidate, player) searches still needed as task sets), the
// searches, and the mask and pawn words.  They differ only in where a state's tasks go:
//   legal_mask_kernel<kLanes>  (one kernel; aq_legal_mask, and aq_legal_mask_ws up to 4,096 states): to the state's own kLanes lanes
//                          (32 / kLanes states per warp, kLanes in {2, 8, 32} by batch size), dealt round-robin by rank; each lane
//                          runs its flood fills in registers.  The per-state work is a variable number of flood fills (0 .. ~60), so
//                          small batches are bound by the slowest states of a nearly empty machine and want many lanes per state, while
//                          large batches want many states per warp.
//   legal_prepare_kernel + legal_search_kernel  (two-phase, below): to a global task list;
//   the legal warpgroup of the fused leaf-evaluation trunk (gnn_tc2.cu): to a task list in shared memory.
// ------------------------------------------------------------------------------------------
constexpr int kLegalWarps = 4;

template <int kLanes>
__global__ void __launch_bounds__(kLegalWarps * 32)
legal_mask_kernel(const AqState *__restrict__ states, int64_t B, uint32_t *__restrict__ mask, uint8_t *__restrict__ pawn) {
    aq_pdl_trigger();  // a kernel launched programmatically behind this one (the GNN trunk of a leaf evaluation) may start as SMs free up
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t b0 = ((int64_t)blockIdx.x * kLegalWarps + warp) * (32 / kLanes) + lane / kLanes;
    const bool valid = b0 < B;
    const int64_t b = valid ? b0 : B - 1;  // out-of-range lanes shadow the last state and write nothing
    LegalPrep p;
    legal_prepare_state<kLanes>(load_state(states + b), lane, p);
    u64 legalH, legalV;
    legal_search_in_place<kLanes, true>(p, lane, legalH, legalV);
    if ((lane & (kLanes - 1)) == 0 && valid) legal_store(p, legalH, legalV, mask + 8 * b, pawn + 8 * b);
}

// ------------------------------------------------------------------------------------------
// K1, two-phase form (the default above 4,096 states): the searches of ALL states go through one flat task list.
//   legal_prepare_kernel : two lanes per state; the prepare step, then the state's tasks are appended to a global task list (one
//                          warp-aggregated atomicAdd) and the mask is written OPTIMISTICALLY (every gated candidate legal);
//   legal_search_kernel  : persistent warps of 32 search state machines fed from the global list through a cursor: a lane whose
//                          flood fill has finished (goal reached, or nothing new: clear the candidate's mask bit) takes the next
//                          task while the others continue.  Fills that fail explore their whole region and take several times
//                          longer than the ones that succeed; one task per thread left 21 of 32 lanes idle on average (ncu,
//                          profiles/): 408 -> 352 us per 1 M positions.
//                          (The same per-lane state machines for the WITNESS paths of the first kernel -- CTA-local task list,
//                          fill and read-back as stages -- were built and measured: 13 instead of 11 active lanes per instruction, no
//                          gain in time, because lanes in different stages split every round; dropped.)
// The per-state number of searches is 0 .. ~60 with a mean of 2-4, so the one-kernel form spends most of its lanes waiting for the
// slowest state of their warp.  A state whose tasks do not fit the list (capacity 8 per state on average) runs them itself
// (legal_search_in_place) -- results never depend on the capacity.
// task word: state index << 8 | slot | (orient - 1) << 6 | opponent << 7;  kNullTask = hole left by an overflow.
// workspace: [0] number of tasks, [1] the search kernel's cursor, tasks from byte 256.
// ------------------------------------------------------------------------------------------
constexpr uint32_t kNullTask = 0xFFFFFFFFu;
constexpr int64_t kLegalChunk = (int64_t)1 << 23;  // states per launch pair (state index field: 24 bits)

#ifndef AQ_PREP_MIN_CTAS
#define AQ_PREP_MIN_CTAS 6
#endif
__global__ void __launch_bounds__(kLegalWarps * 32, AQ_PREP_MIN_CTAS)
legal_prepare_kernel(const AqState *__restrict__ states, int64_t B, uint32_t *__restrict__ mask, uint8_t *__restrict__ pawn,
                     uint32_t *__restrict__ tasks, unsigned cap, unsigned *__restrict__ counter) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane & 1, grp = lane >> 1;
    aq_pdl_trigger();  // legal_search_kernel may be scheduled; it waits for this grid's completion before it reads the task list
    const int64_t b0 = ((int64_t)blockIdx.x * kLegalWarps + warp) * 16 + grp;
    const bool valid = b0 < B;
    const int64_t b = valid ? b0 : B - 1;  // out-of-range lanes shadow the last state and write nothing
    LegalPrep p;
    legal_prepare_state<2>(load_state(states + b), lane, p);
    const int total = valid ? p.offs[4] : 0;
    const unsigned start = legal_reserve(total, lane, counter);  // list space for the whole warp with one atomic
    const bool fits = (u64)start + (unsigned)total <= cap;
    u64 legalH, legalV;
    if (!total || fits) {
        // optimistic: every gated candidate legal (those whose witnesses survive need no search at all);
        // legal_search_kernel clears the bits of the candidates whose search fails
        if (total) legal_for_tasks<2>(p, sub, [&](int i, uint32_t code) { tasks[start + i] = ((uint32_t)b << 8) | code; });
        legalH = p.legalH;
        legalV = p.legalV;
    } else {
        // the list is full: mark what is left of it as holes and run this state's searches here
        for (unsigned t = start + sub; t < cap; t += 2) tasks[t] = kNullTask;
        legal_search_in_place<2, false>(p, lane, legalH, legalV);
    }
    if (sub == 0 && valid) legal_store(p, legalH, legalV, mask + 8 * b, pawn + 8 * b);
}

#ifndef AQ_SEARCH_MIN_CTAS
#define AQ_SEARCH_MIN_CTAS 8
#endif
__global__ void __launch_bounds__(128, AQ_SEARCH_MIN_CTAS)
legal_search_kernel(const AqState *__restrict__ states, const uint32_t *tasks, const unsigned *counter, unsigned *cursor,
                    unsigned cap, uint32_t *__restrict__ mask) {
    aq_pdl_trigger();
    aq_pdl_wait();  // launched programmatically behind legal_prepare_kernel: its task list and counter are complete from here on
    const unsigned n = min(__ldcg(counter), cap);  // coherent loads: see the PDL rule in aq_common.cuh
    const int lane = threadIdx.x & 31;
    legal_search_warp(states, mask, n,
                      [&](unsigned k) {
                          unsigned base = 0;
                          if (lane == 0) base = atomicAdd(cursor, k);
                          return __shfl_sync(0xffffffffu, base, 0);
                      },
                      [&](unsigned t, int64_t &b, uint32_t &code) {
                          const uint32_t w = __ldcg(tasks + t);
                          b = w >> 8;
                          code = w & 0xFFu;
                          return w != kNullTask;
                      });
}

// ordered action list (State.legal_actions() order): pawn list, then per slot H before V
__global__ void legal_list_kernel(const uint32_t *__restrict__ mask, const uint8_t *__restrict__ pawn, int64_t B,
                                  int16_t *__restrict__ actions, int16_t *__restrict__ n_actions) {
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const uint32_t *m = mask + 8 * b;
    int16_t *out = actions + (int64_t)AQ_MAX_LEGAL * b;
    const int np = pawn[8 * b];
    // interleaved candidate index c = 2*slot + (0 H | 1 V); lane handles c = lane + 32*k, k<4
    int base = np;
    for (int k = 0; k < 4; ++k) {
        const int c = lane + 32 * k;
        const int slot = c >> 1;
        const int a = (c & 1) ? (AQ_SQUARES + AQ_SLOTS + slot) : (AQ_SQUARES + slot);
        const bool on = (m[a >> 5] >> (a & 31)) & 1;
        const unsigned bal = __ballot_sync(0xffffffffu, on);
        if (on) out[base + __popc(bal & ((1u << lane) - 1))] = (int16_t)a;
        base += __popc(bal);
    }
    for (int k = lane; k < AQ_MAX_LEGAL; k += 32) {
        if (k < np) out[k] = pawn[8 * b + 1 + k];
        else if (k >= base) out[k] = -1;
    }
    if (lane == 0 && n_actions) n_actions[b] = (int16_t)base;
}

// ------------------------------------------------------------------------------------------
// K9 state_next
// ------------------------------------------------------------------------------------------
__global__ void state_next_kernel(const AqState *__restrict__ states, const int16_t *__restrict__ actions, int64_t B,
                                  AqState *__restrict__ out, uint8_t *__restrict__ terminal) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const AqState t = state_after(load_state(states + b), actions[b]);
    store_state(out + b, t);
    if (terminal) terminal[b] = (uint8_t)terminal_flags(t);
}

// ------------------------------------------------------------------------------------------
// Shortest-path distances and the heuristic evaluation of agents.py:22-54 (SURVEY.md section 8f row 4).
//   dist[b] = {shortest_path_bfs(state), shortest_path_bfs(state seen from the enemy)}; the enemy's search runs
//   un-rotated (start 80 - epos, obstacle ppos, goal row 8), which is the 180-degree image of agents.py:46-48.
//   heur[b]  = (dist_enemy - dist_player) / MAX_DIST_FROM_GOAL in float64 (Python's int / int), agents.py:53
//   leaf48[b] = the depth-0 value of agents.alpha_beta (agents.py:69-75) times 48, as an exact integer:
//               is_lose -> -48, is_draw -> 0, else dist_enemy - dist_player.
// One thread per state: two 81-bit flood fills in registers.
// ------------------------------------------------------------------------------------------
constexpr int kMaxDistFromGoal = AQ_PLIES_FOR_DRAW / 2 - 10;  // agents.py:11 with constants.py:19-20 (NUM_WALLS = 10)

__global__ void __launch_bounds__(128)
shortest_paths_kernel(const AqState *__restrict__ states, int64_t B, int16_t *__restrict__ dist, double *__restrict__ heur,
                      int32_t *__restrict__ leaf48) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const AqState s = load_state(states + b);
    const Open o = open_from_walls(s.hwalls, s.vwalls);
    const int me = s.ppos, en = 80 - (int)s.epos;
    const int dp = path_length(o, me, en, goal_row0());
    const int de = path_length(o, en, me, goal_row8());
    if (dist) *reinterpret_cast<short2 *>(dist + 2 * b) = make_short2((short)dp, (short)de);
    if (heur) heur[b] = (double)(de - dp) / (double)kMaxDistFromGoal;
    if (leaf48) {
        const int t = terminal_flags(s);
        leaf48[b] = (t & 1) ? -kMaxDistFromGoal : (t & 2) ? 0 : de - dp;
    }
}

// Negamax backup of one tree level (agents.py:78-86 without the pruning, which does not change the value inside
// the window nor the action chosen at the root -- see agents.py in this package): for parent p with children
// [off[p], off[p+1]) in legal_actions() order, value[p] = max_c -child_value[c] and best[p] = the FIRST child
// attaining it (agents.py:104 uses a strict '>').  Parents with fixed[p] != kNotFixed keep that value (terminal
// nodes, agents.py:69-73).  One warp per parent.
constexpr int32_t kNotFixed = INT32_MIN;

__global__ void negamax_backup_kernel(const int32_t *__restrict__ child_value, const int64_t *__restrict__ off, int64_t P,
                                      const int32_t *__restrict__ fixed, int32_t *__restrict__ value, int32_t *__restrict__ best) {
    const int lane = threadIdx.x & 31;
    const int64_t p = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= P) return;
    if (fixed && fixed[p] != kNotFixed) {
        if (lane == 0) { value[p] = fixed[p]; if (best) best[p] = -1; }
        return;
    }
    const int64_t lo = off[p], hi = off[p + 1];
    int bv = -(1 << 20);  // "-inf" (agents.py:99) that survives the parent's negation; only a node without any legal action keeps it
    int64_t bi = INT64_MAX;
    for (int64_t c = lo + lane; c < hi; c += 32) {
        const int v = -child_value[c];
        if (v > bv) { bv = v; bi = c; }  // ascending c per lane: keeps the first maximum
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const int ov = __shfl_xor_sync(0xffffffffu, bv, d);
        const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, d);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { value[p] = bv; if (best) best[p] = hi > lo ? (int32_t)(bi - lo) : -1; }
}

// ------------------------------------------------------------------------------------------
// K2 build_graph: one warp per board
// ------------------------------------------------------------------------------------------
__device__ __constant__ float kDinv[6] = {0.f, 1.0f, 0.70710678118654752f, 0.57735026918962576f, 0.5f,
                                          0.44721359549995794f};

__global__ void build_graph_kernel(const AqState *__restrict__ states, int64_t B, uint8_t *__restrict__ open_mask,
                                   float *__restrict__ dinv, float *__restrict__ x, int32_t *__restrict__ edge_count) {
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const AqState s = load_state(states + b);
    const Open o = open_from_walls(s.hwalls, s.vwalls);
    const B81 eh = expand8to9(s.hwalls), ev = expand8to9(s.vwalls);
    int edges = 0;
    for (int v = lane; v < AQ_SQUARES; v += 32) {
        const int m = (int)has(o.up, v) | ((int)has(o.down, v) << 1) | ((int)has(o.left, v) << 2) | ((int)has(o.right, v) << 3);
        edges += __popc(m);
        if (open_mask) open_mask[b * AQ_SQUARES + v] = (uint8_t)m;
        if (dinv) dinv[b * AQ_SQUARES + v] = kDinv[1 + __popc(m)];
        if (x) {
            float2 *px = reinterpret_cast<float2 *>(x + (b * AQ_SQUARES + v) * AQ_FEATURES);
            px[0] = make_float2(v == s.ppos ? 1.f : 0.f, (float)s.pwalls);
            px[1] = make_float2(v == s.epos ? 1.f : 0.f, (float)s.ewalls);  // enemy's own frame, quirk KA11
            px[2] = make_float2(has(eh, v) ? 1.f : 0.f, has(ev, v) ? 1.f : 0.f);
        }
    }
    if (edge_count) {
        edges = __reduce_add_sync(0xffffffffu, edges);
        if (lane == 0) edge_count[b] = edges;
    }
}

__global__ void build_edge_index_kernel(const uint8_t *__restrict__ open_mask, const int64_t *__restrict__ edge_offset,
                                        int64_t B, int64_t *__restrict__ src, int64_t *__restrict__ dst) {
    // one warp per board; canonical order: node ascending, directions U,D,L,R
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    int64_t base = edge_offset[b];
    const int delta[4] = {-9, 9, -1, 1};
    for (int v0 = 0; v0 < 96; v0 += 32) {
        const int v = v0 + lane;
        const int m = v < AQ_SQUARES ? open_mask[b * AQ_SQUARES + v] : 0;
        const int cnt = __popc(m);
        // exclusive prefix over lanes
        int pre = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, pre, d);
            if (lane >= d) pre += t;
        }
        const int tot = __shfl_sync(0xffffffffu, pre, 31);
        int64_t at = base + pre - cnt;
#pragma unroll
        for (int d = 0; d < 4; ++d)
            if ((m >> d) & 1) {
                src[at] = b * AQ_SQUARES + v;
                dst[at] = b * AQ_SQUARES + v + delta[d];
                ++at;
            }
        base += tot;
    }
}

__global__ void edges_to_open_mask_kernel(const int64_t *__restrict__ src, const int64_t *__restrict__ dst, int64_t E,
                                          int64_t B, unsigned *__restrict__ open_words, int32_t *__restrict__ bad) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    const int64_t s = src[e], t = dst[e];
    if (s == t) return;  // self loops are dropped by gcn_norm and re-added
    const int64_t b = s / AQ_SQUARES;
    const int v = (int)(s - b * AQ_SQUARES), u = (int)(t - b * AQ_SQUARES);
    int d = -1;
    if (s >= 0 && b < B && t / AQ_SQUARES == b && t >= 0) {
        const int diff = u - v;
        if (diff == -9) d = 0;
        else if (diff == 9) d = 1;
        else if (diff == -1 && v % AQ_N != 0) d = 2;
        else if (diff == 1 && v % AQ_N != AQ_N - 1) d = 3;
    }
    if (d < 0) { atomicMax(bad, 1); return; }
    // byte v of board b inside a word array (4 bytes per word)
    const int64_t byte = b * AQ_SQUARES + v;
    atomicOr(open_words + (byte >> 2), (1u << d) << (8 * (int)(byte & 3)));
}

// GCNConv normalises with the in-degree at the TARGET node (gcn_norm, flow = source_to_target); the kernels use the degree
// 1 + popcount(open directions) of the node itself.  The two agree exactly when every edge has its reverse, which holds for every
// board graph (is_wall_blocking is symmetric, game_logic.py:145-167).  A caller-supplied edge_index that is not symmetric would be
// evaluated differently from GCNConv, so it is rejected: bad[0] = 2.
__global__ void open_mask_symmetry_kernel(const uint8_t *__restrict__ open_mask, int64_t B, int32_t *__restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * AQ_SQUARES) return;
    const int m = open_mask[i];
    const int delta[4] = {-9, 9, -1, 1};
#pragma unroll
    for (int d = 0; d < 4; ++d)
        if (((m >> d) & 1) && !((open_mask[i + delta[d]] >> (d ^ 1)) & 1)) atomicMax(bad, 2);
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
static inline cudaStream_t S(void *s) { return reinterpret_cast<cudaStream_t>(s); }
static inline unsigned blocks_for(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }

extern "C" int aq_pack_states(const uint8_t *rows68, const int16_t *plies, int64_t B, AqState *out, void *stream) {
    if (B < 0 || (B > 0 && (!rows68 || !out))) return aq_set_error(AQ_ERR_ARG, "aq_pack_states");
    if (B == 0) return 0;
    return aq_launch("aq_pack_states", pack_states_kernel, blocks_for(B, 8), 256, 0, S(stream), false, rows68, plies, B, out);
}

extern "C" int aq_unpack_states(const AqState *states, int64_t B, uint8_t *rows68, int16_t *plies, void *stream) {
    if (B < 0 || (B > 0 && (!rows68 || !states))) return aq_set_error(AQ_ERR_ARG, "aq_unpack_states");
    if (B == 0) return 0;
    return aq_launch("aq_unpack_states", unpack_states_kernel, blocks_for(B, 8), 256, 0, S(stream), false, states, B, rows68, plies);
}

static inline size_t legal_task_cap(int64_t B) { const int64_t n = B < kLegalChunk ? B : kLegalChunk; return (size_t)(8 * n + 4096); }
extern "C" int64_t aq_legal_mask_ws_bytes(int64_t B) { return B <= 0 ? 256 : (int64_t)(256 + 4 * legal_task_cap(B)); }

// ws == NULL: the one-kernel form (lanes per state by batch size); else the two-phase form.
extern "C" int aq_legal_mask_ws(const AqState *states, int64_t B, uint32_t *mask, uint8_t *pawn, void *ws, int64_t ws_bytes,
                                void *stream) {
    if (B < 0 || (B > 0 && (!states || !mask || !pawn))) return aq_set_error(AQ_ERR_ARG, "aq_legal_mask");
    if (B == 0) return 0;
    // measured on B200 (scripts/legal_lanes.py, profiles/): up to 4,096 states one kernel with many lanes per state has the
    // shorter critical path; above, the two-phase form wins
    if (!ws || B <= 4096) {
        const int lanes = B <= 1024 ? 32 : B <= 16384 ? 8 : 2;
        if (lanes == 32)
            return aq_launch("aq_legal_mask", legal_mask_kernel<32>, blocks_for(B, kLegalWarps * 1), kLegalWarps * 32, 0, S(stream), false,
                             states, B, mask, pawn);
        if (lanes == 8)
            return aq_launch("aq_legal_mask", legal_mask_kernel<8>, blocks_for(B, kLegalWarps * 4), kLegalWarps * 32, 0, S(stream), false,
                             states, B, mask, pawn);
        return aq_launch("aq_legal_mask", legal_mask_kernel<2>, blocks_for(B, kLegalWarps * 16), kLegalWarps * 32, 0, S(stream), false,
                         states, B, mask, pawn);
    }
    // any workspace >= 4 KB + 256 B works (a state whose searches do not fit the list runs them itself); aq_legal_mask_ws_bytes(B)
    // is the size at which that practically never happens
    if (ws_bytes < 256 + 4096 || (reinterpret_cast<uintptr_t>(ws) & 3)) return aq_set_error(AQ_ERR_ARG, "aq_legal_mask(workspace)");
    unsigned *counter = reinterpret_cast<unsigned *>(ws);   // [0] task count, [1] the search kernel's cursor
    uint32_t *tasks = reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(ws) + 256);
    const unsigned cap = (unsigned)std::min<int64_t>((ws_bytes - 256) / 4, (int64_t)legal_task_cap(B));
    for (int64_t lo = 0; lo < B; lo += kLegalChunk) {
        const int64_t n = B - lo < kLegalChunk ? B - lo : kLegalChunk;
        cudaError_t e = cudaMemsetAsync(counter, 0, 2 * sizeof(unsigned), S(stream));
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_legal_mask(memset)");
        int rc = aq_launch("aq_legal_mask(prepare)", legal_prepare_kernel, blocks_for(n, kLegalWarps * 16), kLegalWarps * 32, 0, S(stream),
                           false, states + lo, n, mask + 8 * lo, pawn + 8 * lo, tasks, cap, counter);
        if (rc) return rc;
        // persistent warps fed through the cursor: enough of them for the expected number of searches (2-4 per state), at most 8 CTAs
        // of 128 threads per SM
        const unsigned grid = (unsigned)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (3 * n + 127) / 128));
        rc = aq_launch("aq_legal_mask", legal_search_kernel, grid, 128, 0, S(stream), true, states + lo, (const uint32_t *)tasks,
                       (const unsigned *)counter, counter + 1, cap, mask + 8 * lo);
        if (rc) return rc;
    }
    return 0;
}

// State.legal_actions() without a workspace: the one-kernel form (no allocation inside the library).
extern "C" int aq_legal_mask(const AqState *states, int64_t B, uint32_t *mask, uint8_t *pawn, void *stream) {
    return aq_legal_mask_ws(states, B, mask, pawn, nullptr, 0, stream);
}

extern "C" int aq_legal_actions_list(const uint32_t *mask, const uint8_t *pawn, int64_t B, int16_t *actions,
                                     int16_t *n_actions, void *stream) {
    if (B < 0 || (B > 0 && (!mask || !pawn || !actions))) return aq_set_error(AQ_ERR_ARG, "aq_legal_actions_list");
    if (B == 0) return 0;
    return aq_launch("aq_legal_actions_list", legal_list_kernel, blocks_for(B, 8), 256, 0, S(stream), false, mask, pawn, B, actions, n_actions);
}

extern "C" int aq_state_next(const AqState *states, const int16_t *actions, int64_t B, AqState *out, uint8_t *terminal,
                             void *stream) {
    if (B < 0 || (B > 0 && (!states || !actions || !out))) return aq_set_error(AQ_ERR_ARG, "aq_state_next");
    if (B == 0) return 0;
    return aq_launch("aq_state_next", state_next_kernel, blocks_for(B, 256), 256, 0, S(stream), false, states, actions, B, out, terminal);
}

extern "C" int aq_build_graph(const AqState *states, int64_t B, uint8_t *open_mask, float *dinv, float *x,
                              int32_t *edge_count, void *stream) {
    if (B < 0 || (B > 0 && !states)) return aq_set_error(AQ_ERR_ARG, "aq_build_graph");
    if (B == 0) return 0;
    return aq_launch("aq_build_graph", build_graph_kernel, blocks_for(B, 8), 256, 0, S(stream), false, states, B, open_mask, dinv, x,
                     edge_count);
}

extern "C" int aq_build_edge_index(const uint8_t *open_mask, const int64_t *edge_offset, int64_t B, int64_t *src,
                                   int64_t *dst, void *stream) {
    if (B < 0 || (B > 0 && (!open_mask || !edge_offset || !src || !dst)))
        return aq_set_error(AQ_ERR_ARG, "aq_build_edge_index");
    if (B == 0) return 0;
    return aq_launch("aq_build_edge_index", build_edge_index_kernel, blocks_for(B, 8), 256, 0, S(stream), false, open_mask, edge_offset, B,
                     src, dst);
}

extern "C" int aq_edges_to_open_mask(const int64_t *src, const int64_t *dst, int64_t E, int64_t B, uint8_t *open_mask,
                                     int32_t *bad, void *stream) {
    if (B < 0 || E < 0 || !open_mask || !bad || (E > 0 && (!src || !dst)))
        return aq_set_error(AQ_ERR_ARG, "aq_edges_to_open_mask");
    // open_mask must be 4-byte aligned and padded to a multiple of 4 bytes (caller allocates B*81 rounded up)
    if ((reinterpret_cast<uintptr_t>(open_mask) & 3) != 0) return aq_set_error(AQ_ERR_ARG, "aq_edges_to_open_mask(align)");
    cudaError_t e = cudaMemsetAsync(open_mask, 0, (size_t)((B * AQ_SQUARES + 3) / 4 * 4), S(stream));
    if (e != cudaSuccess) return aq_set_error((int)e, "aq_edges_to_open_mask");
    e = cudaMemsetAsync(bad, 0, sizeof(int32_t), S(stream));
    if (e != cudaSuccess) return aq_set_error((int)e, "aq_edges_to_open_mask");
    if (E == 0) return 0;
    const int rc = aq_launch("aq_edges_to_open_mask", edges_to_open_mask_kernel, blocks_for(E, 256), 256, 0, S(stream), false, src, dst, E, B,
                             reinterpret_cast<unsigned *>(open_mask), bad);
    if (rc) return rc;
    return aq_launch("aq_edges_to_open_mask(symmetry)", open_mask_symmetry_kernel, blocks_for(B * AQ_SQUARES, 256), 256, 0, S(stream), false,
                     open_mask, B, bad);
}

extern "C" int aq_shortest_paths(const AqState *states, int64_t B, int16_t *dist, double *heuristic, int32_t *leaf48,
                                 void *stream) {
    if (B < 0 || (B > 0 && (!states || (!dist && !heuristic && !leaf48)))) return aq_set_error(AQ_ERR_ARG, "aq_shortest_paths");
    if (B == 0) return 0;
    return aq_launch("aq_shortest_paths", shortest_paths_kernel, blocks_for(B, 128), 128, 0, S(stream), false, states, B, dist, heuristic,
                     leaf48);
}

extern "C" int aq_negamax_backup(const int32_t *child_value, const int64_t *child_offset, int64_t P, const int32_t *fixed,
                                 int32_t *value, int32_t *best, void *stream) {
    if (P < 0 || (P > 0 && (!child_offset || !value))) return aq_set_error(AQ_ERR_ARG, "aq_negamax_backup");
    if (P == 0) return 0;
    return aq_launch("aq_negamax_backup", negamax_backup_kernel, blocks_for(P, 8), 256, 0, S(stream), false, child_value, child_offset, P,
                     fixed, value, best);
}
