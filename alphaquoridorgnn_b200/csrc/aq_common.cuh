// Shared device helpers: packed state, 81-bit square bitboards, 64-bit wall-slot bitboards.
// Board geometry follows game_logic.py: squares row-major idx = 9*row + col, wall slot
// s = 8*row + col is the 2x2 block whose top-left tile is (row, col)  (game_logic.py:17-19).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/aqgnn.h"

typedef unsigned __int128 u128;
typedef unsigned long long u64;

#define AQ_DEV __host__ __device__ __forceinline__

int aq_set_error(int code, const char *what);
int aq_check_launch(const char *what);
int aq_num_sms();  // multiprocessors of the current device (148 if the query fails)

// Programmatic dependent launch (PDL).  A kernel launched by aq_launch with pdl = true may start while its predecessor in the stream is
// still draining; it must call aq_pdl_wait() before it touches anything the predecessor (or anything earlier in the stream) writes, and
// may run a prologue that reads only long-lived inputs (parameters) before that.  A predecessor that calls aq_pdl_trigger() at its start
// lets the dependent grid be scheduled as soon as SM resources free up; without the trigger the dependent starts when the
// predecessor's blocks have exited, as with a normal launch.  Both device calls are no-ops for normally launched kernels.
// RULE: what the predecessor wrote must be read with coherent loads (__ldcg / plain loads through a non-restrict pointer) after
// aq_pdl_wait().  A load through a `const __restrict__` pointer or __ldg() is an invariant (LDG.CONSTANT) load to the compiler and
// gets hoisted ABOVE the wait -- seen in the SASS of legal_search_kernel, which then read the previous call's task count.
#ifdef __CUDACC__
__device__ __forceinline__ void aq_pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
__device__ __forceinline__ void aq_pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
// Every kernel launch of the library: raises the kernel's dynamic shared-memory limit to `smem` when it uses any, launches (with the
// programmatic-stream-serialization attribute when `pdl` is set) and counts the launch.  Returns 0, or the error reported under `what`.
template <typename... KArgs, typename... Args>
static inline int aq_launch(const char *what, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                            Args... args) {
    cudaError_t e = smem > 0 ? cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) : cudaSuccess;
    if (e == cudaSuccess) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid;
        cfg.blockDim = block;
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = pdl ? 1 : 0;
        e = cudaLaunchKernelEx(&cfg, kernel, args...);
    }
    if (e != cudaSuccess) {
        (void)cudaGetLastError();  // the failed call is also this thread's last error: clear it so that the next launch is not blamed
        return aq_set_error((int)e, what);
    }
    return aq_check_launch(what);
}
#endif

namespace aq {

// ---- 81-square bitboards: three 27-bit words, word w = rows 3w .. 3w+2, bit 9 (r % 3) + c -------------------------------------
// (An `unsigned __int128` board costs 4 ALU instructions per AND/OR and 6-8 per shift on a 32-bit machine; three words that hold
// whole rows need 3, and a row shift by +-1 is one shift per word because the open-direction boards never let a bit leave its row.)
struct B81 {
    uint32_t w0, w1, w2;
};
constexpr uint32_t kM27 = 0x7FFFFFFu;
constexpr uint32_t kRowLo = 0x1FFu;            // first row of a word
constexpr uint32_t kCol0W = 1u | (1u << 9) | (1u << 18);
constexpr uint32_t kCol8W = kCol0W << 8;

AQ_DEV B81 b81(uint32_t a, uint32_t b, uint32_t c) { B81 r; r.w0 = a; r.w1 = b; r.w2 = c; return r; }
AQ_DEV B81 operator&(B81 a, B81 b) { return b81(a.w0 & b.w0, a.w1 & b.w1, a.w2 & b.w2); }
AQ_DEV B81 operator|(B81 a, B81 b) { return b81(a.w0 | b.w0, a.w1 | b.w1, a.w2 | b.w2); }
AQ_DEV B81 andn(B81 a, B81 b) { return b81(a.w0 & ~b.w0, a.w1 & ~b.w1, a.w2 & ~b.w2); }  // a & ~b
AQ_DEV bool any(B81 a) { return (a.w0 | a.w1 | a.w2) != 0u; }
AQ_DEV bool meets(B81 a, B81 b) { return ((a.w0 & b.w0) | (a.w1 & b.w1) | (a.w2 & b.w2)) != 0u; }
AQ_DEV bool same(B81 a, B81 b) { return ((a.w0 ^ b.w0) | (a.w1 ^ b.w1) | (a.w2 ^ b.w2)) == 0u; }
AQ_DEV B81 bit81(int sq) {
    const int w = sq >= 54 ? 2 : sq >= 27 ? 1 : 0;
    const uint32_t m = 1u << (sq - 27 * w);
    return b81(w == 0 ? m : 0u, w == 1 ? m : 0u, w == 2 ? m : 0u);
}
AQ_DEV bool has(B81 b, int sq) {
    const int w = sq >= 54 ? 2 : sq >= 27 ? 1 : 0;
    const uint32_t x = w == 0 ? b.w0 : w == 1 ? b.w1 : b.w2;
    return ((x >> (sq - 27 * w)) & 1u) != 0u;
}
// every square one row down (sq + 9) / up (sq - 9); bits that leave the board are dropped
AQ_DEV B81 down9(B81 b) { return b81((b.w0 << 9) & kM27, ((b.w1 << 9) | (b.w0 >> 18)) & kM27, ((b.w2 << 9) | (b.w1 >> 18)) & kM27); }
AQ_DEV B81 up9(B81 b) { return b81((b.w0 >> 9) | ((b.w1 << 18) & kM27), (b.w1 >> 9) | ((b.w2 << 18) & kM27), b.w2 >> 9); }
// sq + 1 / sq - 1 inside the words (callers mask the source so that no bit crosses a row end)
AQ_DEV B81 right1(B81 b) { return b81((b.w0 << 1) & kM27, (b.w1 << 1) & kM27, (b.w2 << 1) & kM27); }
AQ_DEV B81 left1(B81 b) { return b81(b.w0 >> 1, b.w1 >> 1, b.w2 >> 1); }
AQ_DEV int lowest_square(B81 b) {
#ifdef __CUDA_ARCH__
    return b.w0 ? __ffs((int)b.w0) - 1 : b.w1 ? 27 + __ffs((int)b.w1) - 1 : 54 + __ffs((int)b.w2) - 1;
#else
    return b.w0 ? __builtin_ctz(b.w0) : b.w1 ? 27 + __builtin_ctz(b.w1) : 54 + __builtin_ctz(b.w2);
#endif
}
AQ_DEV int count81(B81 b) {
#ifdef __CUDA_ARCH__
    return __popc(b.w0) + __popc(b.w1) + __popc(b.w2);
#else
    return __builtin_popcount(b.w0) + __builtin_popcount(b.w1) + __builtin_popcount(b.w2);
#endif
}

constexpr u64 kC0 = 0x0101010101010101ull;  // wall-slot column 0
constexpr u64 kC7 = 0x8080808080808080ull;  // wall-slot column 7
constexpr u64 kR0 = 0x00000000000000FFull;  // wall-slot row 0
constexpr u64 kR7 = 0xFF00000000000000ull;  // wall-slot row 7

// 8x8 slot board -> 9x9 square board, slot (x,y) -> square (x,y) (its top-left tile)
AQ_DEV B81 expand8to9(u64 b) {
    const uint32_t lo = (uint32_t)b, hi = (uint32_t)(b >> 32);
    return b81((lo & 0xFFu) | ((lo & 0xFF00u) << 1) | ((lo & 0xFF0000u) << 2),
               (lo >> 24) | ((hi & 0xFFu) << 9) | ((hi & 0xFF00u) << 10),
               ((hi >> 16) & 0xFFu) | ((hi >> 24) << 9));
}
// 9x9 square board -> 8x8 slot board: slot (x,y) <- square (x,y); column 8 and row 8 are dropped
AQ_DEV u64 compress9to8(B81 b) {
    const uint32_t lo = (b.w0 & 0xFFu) | ((b.w0 >> 1) & 0xFF00u) | ((b.w0 >> 2) & 0xFF0000u) | (b.w1 << 24);
    const uint32_t hi = ((b.w1 >> 9) & 0xFFu) | ((b.w1 >> 10) & 0xFF00u) | ((b.w2 & 0xFFu) << 16) | (((b.w2 >> 9) & 0xFFu) << 24);
    return ((u64)hi << 32) | lo;
}

// Open-direction bitboards: bit sq of up/down/left/right set iff the pawn move from sq in that
// direction stays on the board and is not wall-blocked (is_wall_blocking, game_logic.py:145-167).
struct Open {
    B81 up, down, left, right;
};

AQ_DEV Open open_from_walls(u64 h, u64 v) {
    const B81 eh = expand8to9(h), ev = expand8to9(v);
    const B81 bdown = eh | right1(eh);    // H wall in slot (x,y) blocks squares (x,y),(x,y+1) downward
    const B81 bright = ev | down9(ev);    // V wall in slot (x,y) blocks squares (x,y),(x+1,y) rightward
    const B81 bup = down9(bdown), bleft = right1(bright);
    Open o;
    o.down = b81(~bdown.w0 & kM27, ~bdown.w1 & kM27, ~bdown.w2 & (kM27 >> 9));        // no move down from row 8
    o.up = b81(~bup.w0 & (kM27 & ~kRowLo), ~bup.w1 & kM27, ~bup.w2 & kM27);           // none up from row 0
    o.right = b81(~bright.w0 & (kM27 & ~kCol8W), ~bright.w1 & (kM27 & ~kCol8W), ~bright.w2 & (kM27 & ~kCol8W));
    o.left = b81(~bleft.w0 & (kM27 & ~kCol0W), ~bleft.w1 & (kM27 & ~kCol0W), ~bleft.w2 & (kM27 & ~kCol0W));
    return o;
}

// remove the edges severed by one extra wall (o = 1 horizontal, 2 vertical) in slot (x,y)
AQ_DEV void add_wall(Open &o, int orient, int slot) {
    const int x = slot >> 3, y = slot & 7;
    const int sq = 9 * x + y;
    if (orient == 1) {
        const B81 m = bit81(sq) | bit81(sq + 1);
        o.down = andn(o.down, m);
        o.up = andn(o.up, down9(m));
    } else {
        const B81 m = bit81(sq) | bit81(sq + 9);
        o.right = andn(o.right, m);
        o.left = andn(o.left, right1(m));
    }
}

// Targets of a jump over the pawn on `ob` when it is approached moving in direction d
// (0=U,1=D,2=L,3=R): straight if open, else the two perpendicular squares that are open
// (game_logic.py:174-188).  Returned as a bitboard (order is irrelevant for reachability).
AQ_DEV B81 jump_targets(const Open &o, int ob, int d) {
    const bool u = has(o.up, ob), dn = has(o.down, ob), l = has(o.left, ob), r = has(o.right, ob);
    const B81 none = b81(0u, 0u, 0u);
    if (d == 0) return u ? bit81(ob - 9) : ((l ? bit81(ob - 1) : none) | (r ? bit81(ob + 1) : none));
    if (d == 1) return dn ? bit81(ob + 9) : ((l ? bit81(ob - 1) : none) | (r ? bit81(ob + 1) : none));
    if (d == 2) return l ? bit81(ob - 1) : ((u ? bit81(ob - 9) : none) | (dn ? bit81(ob + 9) : none));
    return r ? bit81(ob + 1) : ((u ? bit81(ob - 9) : none) | (dn ? bit81(ob + 9) : none));
}

// The pawn rules around the obstacle square `ob` (the other pawn) for a flood fill: a square from which a move in direction d lands
// on ob (only if that edge is open) is a jump SOURCE; reaching it adds jump_targets(o, ob, d) instead of ob.  The fills keep the
// union of the sources whose jump has not been applied yet (`pending`); a source is reached at most once, so the per-direction
// work below runs at most four times per fill and is recomputed there instead of being carried in registers.
AQ_DEV int jump_source(const Open &o, int ob, int d) {   // -1: no such source
    if (d == 0) return has(o.down, ob) ? ob + 9 : -1;    // below ob, moving up
    if (d == 1) return has(o.up, ob) ? ob - 9 : -1;
    if (d == 2) return has(o.right, ob) ? ob + 1 : -1;   // right of ob, moving left
    return has(o.left, ob) ? ob - 1 : -1;
}
AQ_DEV B81 jump_sources(const Open &o, int ob) {
    B81 p = b81(0u, 0u, 0u);
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        const int s = jump_source(o, ob, d);
        if (s >= 0) p = p | bit81(s);
    }
    return p;
}

// one flood-fill step: the squares reachable by one plain move from `reach`
AQ_DEV B81 step81(const Open &o, B81 reach) {
    return up9(reach & o.up) | down9(reach & o.down) | left1(reach & o.left) | right1(reach & o.right);
}

// bfs() of game_logic.py:309-324 as a bitboard flood fill with the pawn rules of legal_actions_pos applied at every visited
// square: the obstacle square `ob` is never entered; a square adjacent to it (edge open) reaches the jump targets instead.
// The jump rules of one fill, computed once when the fill starts: in a warp that runs 32 fills as per-lane state machines the
// branch that applies a jump is taken by one or two lanes at a time, so it has to be a handful of instructions, not the
// derivation of the targets (measured: deriving them inside the branch halved the lanes active per instruction).
struct Jumps {
    B81 src[4];    // one-hot source square per approach direction (empty: no such source)
    B81 jump[4];   // where a move from that source ends up
};
AQ_DEV Jumps jumps_around(const Open &o, int ob) {
    Jumps j;
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        const int s = jump_source(o, ob, d);
        j.src[d] = s >= 0 ? bit81(s) : b81(0u, 0u, 0u);
        j.jump[d] = jump_targets(o, ob, d);
    }
    return j;
}
struct Fill {
    B81 reach, pending;
    Jumps j;
};
AQ_DEV Fill fill_begin(const Open &o, int start, int ob) {
    Fill f;
    f.reach = bit81(start);
    f.j = jumps_around(o, ob);
    f.pending = (f.j.src[0] | f.j.src[1]) | (f.j.src[2] | f.j.src[3]);
    return f;
}
// One BFS layer.  Returns false when nothing new was reached (the fill is complete).
AQ_DEV bool fill_step(const Open &o, int ob, B81 ob_b, Fill &f) {
    B81 nxt = f.reach | andn(step81(o, f.reach), ob_b);
    if (meets(f.reach, f.pending)) {  // at most four times per fill: a source square was reached, its jump targets join
#pragma unroll
        for (int d = 0; d < 4; ++d)
            if (meets(f.reach, f.j.src[d])) nxt = nxt | f.j.jump[d];
        f.pending = andn(f.pending, f.reach);
    }
    const bool grew = !same(nxt, f.reach);
    f.reach = nxt;
    return grew;
}
// Number of fill iterations (= BFS depth, a jump is one step) after which a square of `goal` is reached, -1 if none is.
AQ_DEV int flood_depth(const Open &o, int start, int ob, B81 goal) {
    Fill f = fill_begin(o, start, ob);
    const B81 ob_b = bit81(ob);
    for (int depth = 0;; ++depth) {
        if (meets(f.reach, goal)) return depth;
        if (!fill_step(o, ob, ob_b, f)) return -1;
    }
}
AQ_DEV bool reaches(const Open &o, int start, int ob, B81 goal) { return flood_depth(o, start, ob, goal) >= 0; }
// shortest_path_bfs of agents.py:27-41: number of pawn steps from `start` to the nearest square of `goal`; -1 if no path (agents.py:41)
AQ_DEV int path_length(const Open &o, int start, int ob, B81 goal) { return flood_depth(o, start, ob, goal); }

AQ_DEV B81 goal_row0() { return b81(kRowLo, 0u, 0u); }
AQ_DEV B81 goal_row8() { return b81(0u, 0u, kRowLo << 18); }

// ---- path witness --------------------------------------------------------------------------------
// One concrete path start -> goal (with the pawn rules) found by the same flood fill, returned as the
// set of wall slots whose H / V wall would sever one of the unit edges the path uses.  A candidate
// wall outside these sets leaves the path intact, so the goal stays reachable and no search is needed:
// walls only ADD blocks, every "edge open" condition the path relies on stays true unless that edge is
// severed, and every "straight jump blocked" condition stays true.  (The converse is not used: a
// candidate that cuts the witness gets a real search.  If no path exists without the candidate, all
// candidates are searched -- a wall behind the other pawn can create diagonal jumps.)
// The fill records for every square the move that reached it first as two direction-code planes (0 = up, 1 = down, 2 = left,
// 3 = right) plus a "by a jump" plane; the path is read back from the goal with one-square lookups.
// The pieces are step functions so that the kernels can run many witnesses per warp as per-lane state machines
// (board_kernels.cu); find_path_cuts() below is the plain loop over the same steps.
struct PathCuts {
    u64 cutH, cutV;
    int exists;
};

AQ_DEV void mark(B81 &b, int sq) {
    const int w = sq >= 54 ? 2 : sq >= 27 ? 1 : 0;
    const uint32_t m = 1u << (sq - 27 * w);
    b.w0 |= w == 0 ? m : 0u; b.w1 |= w == 1 ? m : 0u; b.w2 |= w == 2 ? m : 0u;
}

struct Witness {
    B81 reach, pending;   // the fill
    Jumps j;
    B81 c0, c1, byj;      // first-reached-by planes
    B81 ve, he;           // unit edges of the path read back so far: vertical edge (r,c)-(r+1,c) marked at (r,c) in ve,
                          // horizontal edge (r,c)-(r,c+1) at (r,c) in he
    int cur;              // read-back cursor
};
AQ_DEV Witness witness_begin(const Open &o, int start, int ob) {
    Witness w;
    w.reach = bit81(start);
    w.j = jumps_around(o, ob);
    w.pending = (w.j.src[0] | w.j.src[1]) | (w.j.src[2] | w.j.src[3]);
    w.c0 = w.c1 = w.byj = w.ve = w.he = b81(0u, 0u, 0u);
    w.cur = -1;
    return w;
}
// One BFS layer with the first-reached-by planes.  Returns false when nothing new was reached.
AQ_DEV bool witness_fill_step(const Open &o, int ob, B81 ob_b, Witness &w) {
    const B81 reach = w.reach;
    B81 acc = reach, n;
    n = andn(andn(up9(reach & o.up), ob_b), acc);       acc = acc | n;                                       // code 0
    n = andn(andn(down9(reach & o.down), ob_b), acc);   acc = acc | n; w.c0 = w.c0 | n;                      // code 1
    n = andn(andn(left1(reach & o.left), ob_b), acc);   acc = acc | n; w.c1 = w.c1 | n;                      // code 2
    n = andn(andn(right1(reach & o.right), ob_b), acc); acc = acc | n; w.c0 = w.c0 | n; w.c1 = w.c1 | n;     // code 3
    if (meets(reach, w.pending)) {
#pragma unroll
        for (int d = 0; d < 4; ++d)
            if (meets(reach, w.j.src[d])) {
                n = andn(w.j.jump[d], acc);
                acc = acc | n; w.byj = w.byj | n;
                if (d & 1) w.c0 = w.c0 | n;
                if (d & 2) w.c1 = w.c1 | n;
            }
        w.pending = andn(w.pending, reach);
    }
    const bool grew = !same(acc, reach);
    w.reach = acc;
    return grew;
}
// One step of the read-back from w.cur towards `start`; marks the unit edge(s) of the move that reached w.cur.
AQ_DEV void witness_back_step(int ob, Witness &w) {
    const int cur = w.cur;
    const int code = (int)has(w.c0, cur) | ((int)has(w.c1, cur) << 1);
    const int back = code == 0 ? 9 : code == 1 ? -9 : code == 2 ? 1 : -1;  // from the square back to where the move came from
    if (has(w.byj, cur)) {  // jump over the pawn on ob, approached in direction `code`: unit edges src-ob and ob-cur
        const int src = ob + back;
        if (back == 9 || back == -9) mark(w.ve, src < ob ? src : ob); else mark(w.he, src < ob ? src : ob);
        const int lo = cur < ob ? cur : ob, df = cur < ob ? ob - cur : cur - ob;
        if (df == 9) mark(w.ve, lo); else mark(w.he, lo);
        w.cur = src;
    } else {
        const int prev = cur + back;
        if (back == 9 || back == -9) mark(w.ve, prev < cur ? prev : cur); else mark(w.he, prev < cur ? prev : cur);
        w.cur = prev;
    }
}
// vertical edge at (r,c): H walls in slots (r,c) [c < 8] and (r,c-1) [c > 0]; horizontal edge at (r,c): V walls in slots
// (r,c) [r < 8] and (r-1,c) [r > 0].  compress9to8 drops column 8 / row 8, the shifts drop column 0 / row 0.
AQ_DEV PathCuts witness_cuts(const Witness &w) {
    PathCuts pc;
    pc.exists = 1;
    pc.cutH = compress9to8(w.ve) | compress9to8(left1(andn(w.ve, b81(kCol0W, kCol0W, kCol0W))));
    pc.cutV = compress9to8(w.he) | compress9to8(up9(w.he));
    return pc;
}

AQ_DEV PathCuts find_path_cuts(const Open &o, int start, int ob, B81 goal) {
    Witness w = witness_begin(o, start, ob);
    const B81 ob_b = bit81(ob);
    PathCuts none;
    none.cutH = 0; none.cutV = 0; none.exists = 0;
    while (!meets(w.reach, goal))
        if (!witness_fill_step(o, ob, ob_b, w)) return none;  // goal unreachable even without a candidate
    w.cur = lowest_square(w.reach & goal);
    while (w.cur != start) witness_back_step(ob, w);
    return witness_cuts(w);
}

// legal_actions_pos (game_logic.py:120-192) from square p with the enemy pawn on e (mover's
// frame); writes up to 5 squares in the reference order, returns the count.
AQ_DEV int pawn_moves(const Open &o, int p, int e, uint8_t *out) {
    int n = 0;
    const int delta[4] = {-9, 9, -1, 1};
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        const B81 od = d == 0 ? o.up : d == 1 ? o.down : d == 2 ? o.left : o.right;
        if (!has(od, p)) continue;
        const int q = p + delta[d];
        if (q != e) { out[n++] = (uint8_t)q; continue; }
        if (has(od, q)) { out[n++] = (uint8_t)(q + delta[d]); continue; }
        if (d < 2) {
            if (has(o.left, q)) out[n++] = (uint8_t)(q - 1);
            if (has(o.right, q)) out[n++] = (uint8_t)(q + 1);
        } else {
            if (has(o.up, q)) out[n++] = (uint8_t)(q - 9);
            if (has(o.down, q)) out[n++] = (uint8_t)(q + 9);
        }
    }
    return n;
}

// ---- wall-slot (8x8) neighbourhood shifts: value at slot s taken from its W/E/N/S neighbour --
AQ_DEV u64 fromW(u64 b) { return (b & ~kC7) << 1; }  // s-1, needs col > 0
AQ_DEV u64 fromE(u64 b) { return (b & ~kC0) >> 1; }  // s+1, needs col < 7
AQ_DEV u64 fromN(u64 b) { return b << 8; }           // s-8, needs row > 0
AQ_DEV u64 fromS(u64 b) { return b >> 8; }           // s+8, needs row < 7

struct WallSets {
    u64 freeH, freeV;  // can_place_wall true and the gate does NOT fire -> legal without search
    u64 needH, needV;  // can_place_wall true and the gate fires -> needs both searches
};

// can_place_wall (game_logic.py:199-223) and is_goal_possibly_blocked (227-307) for all 64
// slots and both orientations at once.
AQ_DEV WallSets wall_sets(u64 h, u64 v) {
    const u64 occ = h | v;
    const u64 canH = ~occ & ~fromW(h) & ~fromE(h);
    const u64 canV = ~occ & ~fromN(v) & ~fromS(v);
    // horizontal candidate: left end, middle, right end
    const u64 lH = kC0 | fromW(v) | fromW(fromN(v)) | fromW(fromS(v)) | fromW(fromW(h));
    const u64 mH = fromN(v) | fromS(v);
    const u64 rH = kC7 | fromE(v) | fromE(fromN(v)) | fromE(fromS(v)) | fromE(fromE(h));
    const u64 gateH = (lH & mH) | (lH & rH) | (mH & rH);
    // vertical candidate: top end, middle, bottom end
    const u64 tV = kR0 | fromN(h) | fromN(fromW(h)) | fromN(fromE(h)) | fromN(fromN(v));
    const u64 mV = fromW(h) | fromE(h);
    const u64 bV = kR7 | fromS(h) | fromS(fromW(h)) | fromS(fromE(h)) | fromS(fromS(v));
    const u64 gateV = (tV & mV) | (tV & bV) | (mV & bV);
    WallSets w;
    w.freeH = canH & ~gateH;
    w.needH = canH & gateH;
    w.freeV = canV & ~gateV;
    w.needV = canV & gateV;
    return w;
}

__device__ __forceinline__ AqState load_state(const AqState *p) {
    const uint4 a = __ldg(reinterpret_cast<const uint4 *>(p));
    const uint2 b = __ldg(reinterpret_cast<const uint2 *>(p) + 2);
    AqState s;
    s.hwalls = ((u64)a.y << 32) | a.x;
    s.vwalls = ((u64)a.w << 32) | a.z;
    s.ppos = b.x & 0xFF;
    s.pwalls = (b.x >> 8) & 0xFF;
    s.epos = (b.x >> 16) & 0xFF;
    s.ewalls = (b.x >> 24) & 0xFF;
    s.plies = b.y & 0xFFFF;
    s.flags = (b.y >> 16) & 0xFFFF;
    s.reserved = 0;
    return s;
}

// State.next() (game_logic.py:366-391): apply the action, rotate the board 180 degrees
// (rotate_walls = 64-bit bit reversal of each wall bitboard), swap the players, plies + 1.
__device__ __forceinline__ AqState state_after(AqState s, int a) {
    int ppos = s.ppos, pwalls = s.pwalls;
    if (a < AQ_SQUARES) {
        ppos = a;
    } else if (a < AQ_SQUARES + AQ_SLOTS) {
        s.hwalls |= 1ull << (a - AQ_SQUARES);
        pwalls -= 1;
    } else {
        s.vwalls |= 1ull << (a - AQ_SQUARES - AQ_SLOTS);
        pwalls -= 1;
    }
    AqState t;
    t.hwalls = __brevll(s.hwalls);
    t.vwalls = __brevll(s.vwalls);
    t.ppos = s.epos;
    t.pwalls = s.ewalls;
    t.epos = (uint8_t)ppos;
    t.ewalls = (uint8_t)pwalls;
    t.plies = (uint16_t)(s.plies + 1);
    t.flags = 0;
    t.reserved = 0;
    return t;
}
// is_lose (game_logic.py:43-46) | is_draw << 1 (game_logic.py:49-50)
__device__ __forceinline__ int terminal_flags(const AqState &s) {
    return (int)((s.epos / AQ_N) == 0) | ((int)(s.plies >= AQ_PLIES_FOR_DRAW) << 1);
}
__device__ __forceinline__ void store_state(AqState *p, const AqState &s) {
    uint4 x, y;
    x.x = (unsigned)s.hwalls; x.y = (unsigned)(s.hwalls >> 32); x.z = (unsigned)s.vwalls; x.w = (unsigned)(s.vwalls >> 32);
    y.x = (unsigned)s.ppos | ((unsigned)s.pwalls << 8) | ((unsigned)s.epos << 16) | ((unsigned)s.ewalls << 24);
    y.y = (unsigned)s.plies;
    y.z = 0; y.w = 0;
    reinterpret_cast<uint4 *>(p)[0] = x;
    reinterpret_cast<uint4 *>(p)[1] = y;
}

}  // namespace aq
