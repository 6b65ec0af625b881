// Host build of the legal mask's per-state steps: the same device headers (aq_common.cuh and legal_steps.cuh are
// __host__ __device__ where it matters) compiled for the host.  Test-only: lets the CPU suite check the bitboard
// algorithm (flood fill with pawn rules, bit-parallel gate, witness paths and their task sets, the mask and pawn
// packing) against the golden fixtures before any GPU time is spent.  The warp-level plumbing of the kernels (the
// deal of the tasks to lanes, the task lists, the reductions) is covered by the -m gpu tests.
#include <cstring>
#include "../../alphaquoridorgnn_b200/csrc/legal_steps.cuh"
using namespace aq;

extern "C" void emul_pack(const uint8_t *rows, const int16_t *plies, long long B, AqState *out) {
    for (long long b = 0; b < B; ++b) {
        const uint8_t *r = rows + 68 * b;
        AqState s{};
        for (int i = 0; i < 64; ++i) {
            if (r[4 + i] == 1) s.hwalls |= 1ull << i;
            if (r[4 + i] == 2) s.vwalls |= 1ull << i;
        }
        s.ppos = r[0]; s.pwalls = r[1]; s.epos = r[2]; s.ewalls = r[3];
        s.plies = plies ? (uint16_t)plies[b] : 0;
        out[b] = s;
    }
}

// The kernels' steps one after another: wall sets, the two witness paths, the task sets, one search per task (a failed
// search clears its candidate), the packing.
extern "C" void emul_legal_mask(const AqState *states, long long B, uint32_t *mask, uint8_t *pawn) {
    for (long long b = 0; b < B; ++b) {
        const AqState s = states[b];
        const Open base = open_from_walls(s.hwalls, s.vwalls);
        const int me = s.ppos, en = 80 - (int)s.epos;
        WallSets ws{};
        if (s.pwalls > 0) ws = wall_sets(s.hwalls, s.vwalls);
        const PathCuts pc[2] = {find_path_cuts(base, me, en, goal_row0()), find_path_cuts(base, en, me, goal_row8())};
        u64 set[4];
        legal_task_sets(ws, pc, set);
        u64 legal[2] = {ws.freeH | ws.needH, ws.freeV | ws.needV};
        for (int q = 0; q < 4; ++q)
            for (int slot = 0; slot < 64; ++slot)
                if ((set[q] >> slot) & 1) {
                    Open o = base;
                    add_wall(o, (q & 1) + 1, slot);
                    if (!(q >> 1 ? reaches(o, en, me, goal_row8()) : reaches(o, me, en, goal_row0()))) legal[q & 1] &= ~(1ull << slot);
                }
        const LegalWords w = legal_pack(base, me, en, legal[0], legal[1]);
        memcpy(mask + 8 * b, w.mask, sizeof w.mask);
        memcpy(pawn + 8 * b, w.pawn, sizeof w.pawn);
    }
}

extern "C" void emul_open_mask(const AqState *states, long long B, uint8_t *open_mask) {
    for (long long b = 0; b < B; ++b) {
        const Open o = open_from_walls(states[b].hwalls, states[b].vwalls);
        for (int v = 0; v < 81; ++v)
            open_mask[b * 81 + v] = (uint8_t)((int)has(o.up, v) | ((int)has(o.down, v) << 1) | ((int)has(o.left, v) << 2) | ((int)has(o.right, v) << 3));
    }
}

// shortest_paths_kernel's per-state computation (agents.heuristic_eval, agents.py:22-54)
extern "C" void emul_shortest_paths(const AqState *states, long long B, int16_t *dist) {
    for (long long b = 0; b < B; ++b) {
        const AqState s = states[b];
        const Open o = open_from_walls(s.hwalls, s.vwalls);
        const int me = s.ppos, en = 80 - (int)s.epos;
        dist[2 * b] = (int16_t)path_length(o, me, en, goal_row0());
        dist[2 * b + 1] = (int16_t)path_length(o, en, me, goal_row8());
    }
}
