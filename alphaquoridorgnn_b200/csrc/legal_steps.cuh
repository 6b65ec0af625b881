// The per-state steps of the legal mask, shared by all three forms of it, which differ only in where a state's tasks go:
//   legal_mask_kernel<2/8/32>   (board_kernels.cu, one kernel)  the state's own lanes run them in place;
//   legal_prepare_kernel / legal_search_kernel (board_kernels.cu, two-phase)  a global task list;
//   the legal warpgroup of the fused leaf-evaluation trunk (gnn_tc2.cu)  a CTA-local task list in shared memory.
//   prepare : kLanes lanes per state.  Open-direction boards, can_place + gate of all 128 candidates, and the witness paths (sub-lane
//             0: the mover's, sub-lane 1: the opponent's); the (candidate, player) searches still needed are the task sets.
//   search  : in place, the state's tasks dealt round-robin by rank to its lanes; or per-lane flood-fill state machines of one warp,
//             fed from a task list: a lane whose fill has finished (goal reached, or nothing new: clear the candidate's mask bit)
//             takes the next task while the others continue.
// A task code is slot | (orient - 1) << 6 | opponent << 7 (8 bits); the list entry adds the state.
// legal_task_sets and legal_pack are __host__ __device__: the host-side checks of the test suite run them too.
#pragma once
#include "aq_common.cuh"

namespace aq {

// The searches a state still needs (game_logic.py:332-348): a gated candidate is searched for a player only if it cuts that player's
// witness path, and for every gated candidate when the player has no path.  pc = {mover's, opponent's} witness cuts;
// set = [mover H, mover V, opponent H, opponent V].
AQ_DEV void legal_task_sets(const WallSets &ws, const PathCuts pc[2], u64 set[4]) {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        set[2 * q + 0] = ws.needH & (pc[q].exists ? pc[q].cutH : ~0ull);
        set[2 * q + 1] = ws.needV & (pc[q].exists ? pc[q].cutV : ~0ull);
    }
}

// mask [8] u32 and pawn [8] u8 of one state: actions 0..80 the pawn moves, 81..144 the H walls, 145..208 the V walls; the pawn
// moves' count, then up to five squares in the reference order.
struct LegalWords {
    uint32_t mask[8];
    uint32_t pawn[2];
};
AQ_DEV LegalWords legal_pack(const Open &base, int me, int en, u64 legalH, u64 legalV) {
    uint8_t pm[8] = {0, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0, 0};
    const int n = pawn_moves(base, me, en, pm + 1);
    pm[0] = (uint8_t)n;
    u128 lo = 0;
    for (int k = 0; k < n; ++k) lo |= (u128)1 << pm[1 + k];
    lo |= (u128)legalH << 81;                                  // H wall actions 81..144
    const u128 hi = (u128)(legalH >> 47) | ((u128)legalV << 17);  // V wall actions 145..208
    LegalWords w;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        w.mask[k] = (uint32_t)(lo >> (32 * k));
        w.mask[4 + k] = (uint32_t)(hi >> (32 * k));
    }
    w.pawn[0] = pm[0] | (pm[1] << 8) | (pm[2] << 16) | ((unsigned)pm[3] << 24);
    w.pawn[1] = pm[4] | (pm[5] << 8);
    return w;
}

struct LegalPrep {
    Open base;
    int me, en;             // mover's square, enemy square in the mover's frame (game_logic.py:136)
    u64 legalH, legalV;     // legal unless a search of the task sets fails: the free and the gated candidates
    u64 set[4];             // tasks: [mover H, mover V, opponent H, opponent V]
    int offs[5];            // exclusive prefix of the set sizes; offs[4] = the state's number of tasks
};

// Prepare step of state s.  kLanes lanes per state (sub = lane & (kLanes - 1)); every lane of the warp calls it (group shuffles).
template <int kLanes>
__device__ __forceinline__ void legal_prepare_state(const AqState &s, int lane, LegalPrep &p) {
    const int sub = lane & (kLanes - 1);
    p.base = open_from_walls(s.hwalls, s.vwalls);
    p.me = s.ppos; p.en = 80 - (int)s.epos;
    WallSets ws;
    ws.freeH = 0; ws.freeV = 0; ws.needH = 0; ws.needV = 0;
    if (s.pwalls > 0) ws = wall_sets(s.hwalls, s.vwalls);  // game_logic.py:113
    p.legalH = ws.freeH | ws.needH;
    p.legalV = ws.freeV | ws.needV;
    // witness paths: mover (start me, obstacle en, goal row 0) on sub-lane 0, opponent in the un-rotated frame
    // (start en, obstacle me, goal row 8) on sub-lane 1
    PathCuts pc;
    pc.cutH = 0; pc.cutV = 0; pc.exists = 1;
    if (sub < 2 && (ws.needH | ws.needV))
        pc = find_path_cuts(p.base, sub == 0 ? p.me : p.en, sub == 0 ? p.en : p.me, sub == 0 ? goal_row0() : goal_row8());
    __syncwarp();
    PathCuts w[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int src = (lane & ~(kLanes - 1)) | q;
        w[q].exists = __shfl_sync(0xffffffffu, pc.exists, src);
        w[q].cutH = ((u64)__shfl_sync(0xffffffffu, (unsigned)(pc.cutH >> 32), src) << 32) | __shfl_sync(0xffffffffu, (unsigned)pc.cutH, src);
        w[q].cutV = ((u64)__shfl_sync(0xffffffffu, (unsigned)(pc.cutV >> 32), src) << 32) | __shfl_sync(0xffffffffu, (unsigned)pc.cutV, src);
    }
    legal_task_sets(ws, w, p.set);
    p.offs[0] = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) p.offs[q + 1] = p.offs[q] + __popcll(p.set[q]);
}

// List space for the tasks of a warp's 16 states with one atomic on `counter`: exclusive scan of the per-state totals (held by
// both lanes of a pair); returns the first entry of this state's range.
__device__ __forceinline__ unsigned legal_reserve(int total, int lane, unsigned *counter) {
    const int sub = lane & 1;
    int incl = sub == 0 ? total : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    const int warp_total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned wbase = 0;
    if (lane == 0 && warp_total) wbase = atomicAdd(counter, (unsigned)warp_total);
    wbase = __shfl_sync(0xffffffffu, wbase, 0);
    return wbase + (unsigned)__shfl_sync(0xffffffffu, incl - (sub == 0 ? total : 0), lane & ~1);
}

// The lane's share of the state's tasks: f(i, code) for every task whose rank i among the state's tasks (offs[q] + its rank within
// set q) is sub modulo kLanes, in rank order.  A walk over the set bits, with one call site of f per set (q known at compile time).
template <int kLanes, class F>
__device__ __forceinline__ void legal_for_tasks(const LegalPrep &p, int sub, F f) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        int i = p.offs[q];
        for (u64 mm = p.set[q]; mm; mm &= mm - 1, ++i)
            if ((i & (kLanes - 1)) == sub) f(i, (uint32_t)(((__ffsll((long long)mm) - 1) & 63) | (q << 6)));  // & 63: code >> 6 is q at compile time
    }
}

// The state's lanes run its searches themselves, clear the bits of the candidates whose search fails and AND the legal sets over the
// lane group.  Two ways to split the searches between the lanes, with the same result (the mask is an AND over the same searches):
//   kTogether: every lane of the warp runs its share at the same time (legal_mask_kernel).  Each lane takes the tasks of its rank
//              (legal_for_tasks), collected first and searched from one call site, so that lanes whose tasks lie in different sets
//              fill together.
//   otherwise: the overflow branch of the two-lane task-list forms, taken pair by pair (divergently) by the few states that do not
//              fit the list.  Each lane takes the slots of its parity in each set, a fixed-count loop per set with the set known at
//              compile time: it holds fewer registers across the rest of those kernels, which run with a register cap (the prepare
//              kernel) or beside the trunk (the fused warpgroup); the rank deal put spills into their witness fill loops.
template <int kLanes, bool kTogether>
__device__ __forceinline__ void legal_search_in_place(const LegalPrep &p, int lane, u64 &legalH, u64 &legalV) {
    const int sub = lane & (kLanes - 1);
    legalH = p.legalH;
    legalV = p.legalV;
    auto search = [&](uint32_t code) {
        const int slot = code & 63, orient = ((code >> 6) & 1) + 1, opp = code >> 7;
        Open o = p.base;
        add_wall(o, orient, slot);
        if (!reaches(o, opp ? p.en : p.me, opp ? p.me : p.en, opp ? goal_row8() : goal_row0())) {
            if (orient == 1) legalH &= ~(1ull << slot); else legalV &= ~(1ull << slot);
        }
    };
    if constexpr (kTogether) {
        u64 mine[4] = {0, 0, 0, 0};
        legal_for_tasks<kLanes>(p, sub, [&](int, uint32_t code) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (k == (int)(code >> 6)) mine[k] |= 1ull << (code & 63);
        });
        while (mine[0] | mine[1] | mine[2] | mine[3]) {
            const int q = mine[0] ? 0 : mine[1] ? 1 : mine[2] ? 2 : 3;
            uint32_t code = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (k == q) {
                    code = (uint32_t)(__ffsll((long long)mine[k]) - 1) | (k << 6);
                    mine[k] &= mine[k] - 1;
                }
            search(code);
        }
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q)
            for (int slot = sub; slot < 64; slot += kLanes)
                if ((p.set[q] >> slot) & 1) search((uint32_t)slot | (q << 6));
    }
    const unsigned gmask = (kLanes == 32 ? 0xffffffffu : (1u << (kLanes & 31)) - 1u) << (lane & ~(kLanes - 1));
#pragma unroll
    for (int d = 1; d < kLanes; d <<= 1) {
        legalH &= ((u64)__shfl_xor_sync(gmask, (unsigned)(legalH >> 32), d) << 32) | __shfl_xor_sync(gmask, (unsigned)legalH, d);
        legalV &= ((u64)__shfl_xor_sync(gmask, (unsigned)(legalV >> 32), d) << 32) | __shfl_xor_sync(gmask, (unsigned)legalV, d);
    }
}

// mask [8] u32 and pawn [8] u8 of one state (one lane)
__device__ __forceinline__ void legal_store(const LegalPrep &p, u64 legalH, u64 legalV, uint32_t *mask, uint8_t *pawn) {
    const LegalWords w = legal_pack(p.base, p.me, p.en, legalH, legalV);
    uint4 *m = reinterpret_cast<uint4 *>(mask);
    m[0] = make_uint4(w.mask[0], w.mask[1], w.mask[2], w.mask[3]);
    m[1] = make_uint4(w.mask[4], w.mask[5], w.mask[6], w.mask[7]);
    *reinterpret_cast<uint2 *>(pawn) = make_uint2(w.pawn[0], w.pawn[1]);
}

#ifndef AQ_FILL_STEPS
#define AQ_FILL_STEPS 2
#endif
#ifndef AQ_REFILL_IDLE
#define AQ_REFILL_IDLE 28
#endif
constexpr int kRefillIdle = AQ_REFILL_IDLE;   // a warp fetches new tasks when at least this many of its lanes are idle

// Search step: the n tasks of a list run by one warp together with the other warps that share the list's cursor.
//   claim(k)              reserves k consecutive entries, returns the first (called by every lane; the result is warp-uniform);
//   fetch(t, b, code)     reads entry t < n: false for a hole, else the state index b and the task code.
// A failed search clears its candidate's bit of mask[8 b ..] with atomicAnd (the mask was written optimistically).
template <class Claim, class Fetch>
__device__ __forceinline__ void legal_search_warp(const AqState *states, uint32_t *mask, unsigned n, Claim claim, Fetch fetch) {
    const int lane = threadIdx.x & 31;
    bool active = false, exhausted = n == 0u;
    Open o;
    Fill f;
    B81 ob_b = b81(0u, 0u, 0u), goal = ob_b;
    o.up = o.down = o.left = o.right = ob_b;
    f.reach = f.pending = ob_b;
#pragma unroll
    for (int d = 0; d < 4; ++d) f.j.src[d] = f.j.jump[d] = ob_b;
    int ob = 0, action = 0;
    int64_t b = 0;
    while (true) {
        unsigned act = __ballot_sync(0xffffffffu, active);
        const int n_idle = 32 - __popc(act);
        if (!exhausted && (n_idle >= kRefillIdle || act == 0u)) {
            const unsigned base = claim((unsigned)n_idle);
            exhausted = base + (unsigned)n_idle >= n;
            if (!active) {
                const unsigned t = base + (unsigned)__popc(~act & ((1u << lane) - 1u));
                int64_t tb = 0;
                uint32_t code = 0;
                if (t < n && fetch(t, tb, code)) {
                    b = tb;
                    const int slot = code & 63, orient = ((code >> 6) & 1) + 1, opp = (code >> 7) & 1;
                    const AqState s = load_state(states + b);
                    o = open_from_walls(s.hwalls, s.vwalls);
                    add_wall(o, orient, slot);
                    const int me = s.ppos, en = 80 - (int)s.epos;
                    ob = opp ? me : en;
                    goal = opp ? goal_row8() : goal_row0();
                    ob_b = bit81(ob);
                    f = fill_begin(o, opp ? en : me, ob);
                    action = AQ_SQUARES + (orient == 2 ? AQ_SLOTS : 0) + slot;
                    active = true;
                }
            }
            act = __ballot_sync(0xffffffffu, active);
        }
        if (act == 0u) {
            if (exhausted) break;
            continue;   // every fetched entry was a hole: fetch again
        }
        if (active) {
            // two BFS layers per round (one exit test per two layers: the fill is monotone, a layer too many changes nothing)
            bool grew = fill_step(o, ob, ob_b, f);
#pragma unroll
            for (int k = 1; k < AQ_FILL_STEPS; ++k)
                if (grew && !meets(f.reach, goal)) grew = fill_step(o, ob, ob_b, f);
            if (meets(f.reach, goal)) {
                active = false;
            } else if (!grew) {
                atomicAnd(mask + 8 * b + (action >> 5), ~(1u << (action & 31)));
                active = false;
            }
        }
    }
}

}  // namespace aq
