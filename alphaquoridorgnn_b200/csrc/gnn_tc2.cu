// bf16 tensor-core GCN trunk, version 2 (inference): the node transform AND the A_hat aggregation both run
// on the 5th-gen tensor cores; the CUDA cores only convert accumulators to bf16 and build the per-board
// operands.  Per board  X_{l+1} = ReLU(A_hat (X_l W_l^T) + b_l)  is evaluated feature-major:
//
//   transform   Z^T = W X^T        A = W   [128 out][128 in]  bf16 resident in TENSOR MEMORY (TS form of tcgen05.mma)
//                                  B = X^T [K = 128 feat][N = 96 nodes]  MN-major SWIZZLE_64B in shared memory
//                                  D = Z^T [128 lanes = features][96 columns = nodes]  fp32 in TMEM
//   aggregate   Y^T = Z^T A_hat^T  A = Z^T [M = 128 feat][K = 96 nodes]  K-major SWIZZLE_64B -- byte for byte the same
//                                     "feature-major" tile as the transform's B operand, so one 24 KB buffer per board serves both
//                                  B = A_hat, banded: two blocks of [48 out nodes][64 in nodes] K-major SWIZZLE_128B (a 5-point
//                                      stencil on a 9x9 board reaches at most 9 nodes away: out nodes 0..47 need in nodes 0..63,
//                                      out nodes 48..80 need 32..95)
//                                  the aggregation runs in FP16 (A and B must share a format): the coefficients dinv_i dinv_j
//                                  lie in [0.2, 1] and keep 11 mantissa bits, Z is converted with saturation (|z| <= 65504)
//                                  the bias is added in fp32 by the epilogue (an extra "ones column" MMA step costs shared-memory bandwidth)
//                                  D = Y^T [128 lanes][96 columns]
//
// A thread owns one feature (TMEM lane) of its board; every epilogue is "tcgen05.ld 32 columns -> cvt.bf16x2 / cvt.f16x2 ->
// four 16-byte shared stores into the thread's own tile row": no scattered stores, no stencil arithmetic.  Only the 5
// non-zero positions per adjacency row are rewritten per board (the tiles are zeroed once per kernel).
//
// One persistent CTA per SM, 4 independent 4-warp groups (one board each in flight).  TMEM: 4 x 96 accumulator columns +
// 2 x 64 columns holding W2 and W3 = 512.  Shared memory: 4 x 52 KB group state (tile, double-buffered adjacency,
// layer-1 operand) + shared operands and tables.
//   * Node phase (per board, 81 node threads): open directions from two 18-bit windows of the wall bitboards, degrees exchanged
//     through shared memory, coefficients and their fp16 bits from a 64-entry table, the six input planes from the same windows;
//     it is software-pipelined: the node phase of a group's NEXT board runs while its last aggregation is in flight.
//   * MMAs are issued by the first warp of each group from warp-uniform values (elect.sync inside a uniform branch) so that the
//     descriptors live in uniform registers; issuing from `if (tid == 0)` cost ~80 cycles per MMA (R2UR broadcast loops).
//   * Layer 1 (K = 6): fp32 aggregation of the 6-wide input by the node threads, one K = 16 MMA (hi/lo split input, bias folded),
//     as in version 1 (gnn_tc.cu).
// Measured at B = 16,384 (CUDA events): 251 us (version 1) -> 146 us.  What bounds it now (ncu): the F2FP packs on the XU pipe
// (16 cycles per warp instruction on this part) and shared-memory bandwidth (SS-mode N = 48 MMAs re-read the 4 KB A slice).
#include <cstddef>
#include <cstdlib>
#include <cuda_bf16.h>
#include "gnn_fp32.cuh"
#include "tc_common.cuh"
#include "legal_steps.cuh"

using namespace aq;
using namespace aqtc;

#ifndef TC2_PREFETCH
#define TC2_PREFETCH 1   // 1: fetch the next board's state one board ahead
#endif


#ifndef TC2_TIMING
#define TC2_TIMING 0     // 1: per-phase clock64 accounting by thread 0 of group 0 of CTA 0 (debug variant)
#endif
#if TC2_TIMING
__device__ long long g_tc2_timing[16];
#define TC2_T(slot) do { if (blockIdx.x == 0 && gtid == 0) { const long long t_ = clock64(); g_tc2_timing[slot] += t_ - t_last; t_last = t_; } } while (0)
extern "C" int aq_debug_tc2_timing(long long *out) {
    cudaMemcpyFromSymbol(out, g_tc2_timing, sizeof(long long) * 16);
    long long z[16] = {0};
    cudaMemcpyToSymbol(g_tc2_timing, z, sizeof(z));
    return 0;
}
#else
#define TC2_T(slot) do { } while (0)
#endif

#ifndef TC2_FINISH
#define TC2_FINISH 0     // 1: per-CTA finish stamps of the legal warpgroup and the trunk groups (debug variant, scripts/fused_finish.py)
#endif
#if TC2_FINISH
// per CTA: [0] start (globaltimer ns), [1] legal warpgroup done (ns), [2] last trunk group done (ns), [3] legal warpgroup done
// (SM clock cycles after the start), [4] last trunk group done (cycles), [5] boards of the CTA's first trunk group
constexpr int kFinishCtas = 1024;
__device__ unsigned long long g_tc2_finish[kFinishCtas][8];
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
    return t;
}
extern "C" int aq_debug_tc2_finish(unsigned long long *out) {
    cudaMemcpyFromSymbol(out, g_tc2_finish, sizeof(g_tc2_finish));
    static unsigned long long z[kFinishCtas][8];
    cudaMemcpyToSymbol(g_tc2_finish, z, sizeof(z));
    return kFinishCtas;
}
#endif
#ifndef TC2_OVERFLOW_COUNT
#define TC2_OVERFLOW_COUNT 0   // 1: count the states whose searches did not fit the legal warpgroup's task list (debug variant)
#endif
#if TC2_OVERFLOW_COUNT
__device__ unsigned long long g_tc2_overflow;
extern "C" long long aq_debug_tc2_overflow(void) {
    unsigned long long n = 0, z = 0;
    cudaMemcpyFromSymbol(&n, g_tc2_overflow, sizeof(n));
    cudaMemcpyToSymbol(g_tc2_overflow, &z, sizeof(z));
    return (long long)n;
}
#endif

namespace {

constexpr int kG = 4;             // groups (boards in flight) per CTA
constexpr uint32_t kGroupCols = 96;                  // TMEM columns per group: accumulator [128 x 96] fp32
constexpr int kNodesPad = 96;
constexpr uint32_t kFmBlock = 16 * 512;              // feature-major tile: [3 node blocks of 32][16 atoms of 8 features][8][64 B]
constexpr uint32_t kAdjBlock = 48 * 128;             // adjacency block: 48 out-node rows x 64 in-nodes (128 B)
constexpr uint32_t kWKBlock = 128 * 128;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kTmemW2 = kG * kGroupCols, kTmemW3 = kTmemW2 + 64;
static_assert(kTmemW3 + 64 <= kTmemCols, "TMEM columns");

// instruction descriptors (kind::f16): D = f32, A = B = bf16, M = 128
constexpr uint32_t kIdescBase = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24);
constexpr uint32_t kIdescL1 = kIdescBase | ((uint32_t)(kNodesPad >> 3) << 17);                 // K-major A and B, N = 96
constexpr uint32_t kIdescT = kIdescBase | (1u << 16) | ((uint32_t)(kNodesPad >> 3) << 17);     // B MN-major, N = 96
constexpr uint32_t kIdescA = (1u << 4) | ((128u >> 4) << 24) | ((uint32_t)(48 >> 3) << 17);    // A = B = f16, K-major, N = 48

// Loop-invariant facts about node v = (r, c), built once per CTA.  Wall slots are read through an 18-bit window of the
// H / V bitboards that starts at slot 8 r + c - 9: bit 0 = slot (r-1, c-1), 1 = (r-1, c), 8 = (r, c-1), 9 = (r, c),
// 10 = (r, c+1), 17 = (r+1, c).  Bit 31 of a blocking mask stands for "this direction does not exist".
struct NodeConst {
    uint32_t upm, dnm, lfm, rtm;             // slots whose wall closes the move up / down (H board) and left / right (V board)
    uint32_t pv, sh, adj01, adj23;           // valid wall-plane bits {self 9, up 1, down 17, left 8, right 10}; window shift; tile offsets
    uint32_t adj4, row_off, pad0, pad1;      // ... of the stencil positions self|up, down|left, right (0xFFFF = absent); layer-1 operand row offset
};

struct Tc2Group {
    unsigned char fm[3 * kFmBlock];          // 24 KB: X^T (B operand, MN-major) / Z^T (A operand, K-major)
    unsigned char adj[2][2][kAdjBlock];      // 2 x 12 KB: A_hat (fp16) [board parity][block 0 | 1] -- the next board's tile is built
                                             //            while the current board's last aggregation is still reading its own
    unsigned char l1op[kNodesPad * 32];      // 3 KB: layer-1 node operand [96 nodes][16] K-major SWIZZLE_32B
    uint8_t deg[128];                        // degree (1 + open directions) of node v at [16 + v]; neighbours are read at 16 + v +- 1 / 9
    unsigned char pad[1024 - 128];
};
static_assert(sizeof(Tc2Group) % 1024 == 0, "group state must keep 1024-byte alignment");

struct Tc2Smem {
    unsigned char w1[128 * 32];              // layer-1 weight operand [128][16] K-major SWIZZLE_32B: [W1 | W1 | b1_hi | b1_lo | 0 | 0]
    Tc2Group g[kG];
    NodeConst nc[kV];                        // loop-invariant per-node constants
    float2 lut[64];                          // [deg_v * 8 + deg_u] -> {dinv_v * dinv_u as float, the same as fp16 bits}; entry 0 = closed edge
    unsigned long long mbar[kG];
    uint32_t tmem_base;
};
static_assert(offsetof(Tc2Smem, g) % 1024 == 0, "group state must be 1024-byte aligned");
static_assert(sizeof(Tc2Smem) + 1024 <= 227 * 1024, "Tc2Smem exceeds shared memory");

// Legal warpgroup of the fused leaf evaluation (kLegal): a fifth 4-warp group computes the legal mask of the CTA's boards while the
// four trunk groups run.  Rounds of 64 states: prepare (two lanes per state, legal_steps.cuh) appends the searches to a task list in
// shared memory behind Tc2Smem, then the four warps run them as per-lane search state machines through a shared cursor.
constexpr int kTrunkThreads = kG * kGroupThreads;
constexpr int kLegalThreads = 128;
constexpr int kLegalStates = kLegalThreads / 2;        // states per round
#ifndef TC2_LEGAL_CAP
#define TC2_LEGAL_CAP 2048
#endif
constexpr int kLegalCap = TC2_LEGAL_CAP;               // task entries (32 per state; the mean is 2-4)
constexpr unsigned short kNullTask16 = 0xFFFFu;
struct Tc2Legal {
    unsigned short task[kLegalCap];                    // state within the round << 8 | task code; kNullTask16 = hole left by an overflow
    unsigned count[2][2];                              // [round parity][number of tasks, search cursor]
};
static_assert(sizeof(Tc2Smem) % 8 == 0 && sizeof(Tc2Smem) + sizeof(Tc2Legal) + 1024 <= 227 * 1024, "Tc2Legal exceeds shared memory");
static_assert(kLegalStates <= 256, "state within the round is 8 bits of a task entry");

__device__ __forceinline__ void legal_sync() { asm volatile("bar.sync 5, %0;\n" ::"n"(kLegalThreads) : "memory"); }
__device__ __forceinline__ void trunk_sync() { asm volatile("bar.sync 6, %0;\n" ::"n"(kTrunkThreads) : "memory"); }

// The legal warpgroup: mask [B][8] and pawn [B][8] of the boards b = blockIdx.x * kG + g + k * stride that the CTA's trunk groups
// process (state i of the CTA is board (i & 3) + (i >> 2) * stride past the CTA's first).  lt = thread within the warpgroup.
__device__ __forceinline__ void legal_warpgroup(const AqState *__restrict__ states, int64_t B, uint32_t *mask, uint8_t *pawn, Tc2Legal &L,
                                                int lt) {
    const int lane = lt & 31, sub = lt & 1, j = lt >> 1;
    const int64_t first = (int64_t)blockIdx.x * kG, stride = (int64_t)gridDim.x * kG;
    auto board = [&](int64_t i) { return first + (i & (kG - 1)) + (i >> 2) * stride; };
    if (lt < 4) L.count[lt >> 1][lt & 1] = 0u;
    legal_sync();
    int par = 0;
    for (int64_t i0 = 0; board(i0) < B; i0 += kLegalStates, par ^= 1) {
        // ---- prepare: witness paths, optimistic mask, searches -> the round's task list --------------------------------
        const int64_t b0 = board(i0 + j);
        const bool valid = b0 < B;
        const int64_t b = valid ? b0 : board(i0);  // out-of-range lanes shadow the round's first state and write nothing
        LegalPrep p;
        legal_prepare_state<2>(load_state(states + b), lane, p);
        const int total = valid ? p.offs[4] : 0;
        const unsigned start = legal_reserve(total, lane, &L.count[par][0]);
        u64 legalH, legalV;
        if (!total || start + (unsigned)total <= (unsigned)kLegalCap) {
            if (total) legal_for_tasks<2>(p, sub, [&](int k, uint32_t code) { L.task[start + k] = (unsigned short)((j << 8) | code); });
            legalH = p.legalH;
            legalV = p.legalV;
        } else {  // the list is full: mark what is left of it as holes and run this state's searches here
            for (unsigned t = start + sub; t < (unsigned)kLegalCap; t += 2) L.task[t] = kNullTask16;
            legal_search_in_place<2, false>(p, lane, legalH, legalV);
#if TC2_OVERFLOW_COUNT
            if (sub == 0) atomicAdd(&g_tc2_overflow, 1ull);
#endif
        }
        if (sub == 0 && valid) legal_store(p, legalH, legalV, mask + 8 * b, pawn + 8 * b);
        legal_sync();   // the task list and the optimistic mask words are complete
        // ---- search: the round's tasks through the shared cursor; a failed search clears its mask bit ----------------------
        if (lt == 0) { L.count[par ^ 1][0] = 0u; L.count[par ^ 1][1] = 0u; }  // the next round's counters (last used two rounds ago)
        const unsigned n = min(L.count[par][0], (unsigned)kLegalCap);
        legal_search_warp(states, mask, n,
                          [&](unsigned k) {
                              unsigned base = 0;
                              if (lane == 0) base = atomicAdd(&L.count[par][1], k);
                              return __shfl_sync(0xffffffffu, base, 0);
                          },
                          [&](unsigned t, int64_t &tb, uint32_t &code) {
                              const unsigned w = L.task[t];
                              tb = board(i0 + (w >> 8));
                              code = w & 0xFFu;
                              return w != kNullTask16;
                          });
        legal_sync();   // the task list is free for the next round
    }
}

__device__ __forceinline__ uint64_t desc_fm_mn(uint32_t saddr) {  // MN-major SWIZZLE_64B: LBO = node-block stride, SBO = 8-feature atom stride
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(kFmBlock >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
__device__ __forceinline__ uint64_t desc_fm_k(uint32_t saddr) {   // K-major SWIZZLE_64B: SBO = 512 B (8 rows x 64 B)
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a_tmem, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
                 ::"r"(d), "r"(a_tmem), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t *r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
                 "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
                   "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
                   "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
                   "r"(r[30]), "r"(r[31]) : "memory");
}
// two floats -> packed bf16x2 (a in the low half), optionally through ReLU
template <bool kRelu>
__device__ __forceinline__ uint32_t cvt2(float a, float b) {
    uint32_t d;
    if (kRelu) asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;\n" : "=r"(d) : "f"(b), "f"(a));
    else asm("cvt.rn.bf16x2.f32 %0, %1, %2;\n" : "=r"(d) : "f"(b), "f"(a));
    return d;
}
__device__ __forceinline__ uint32_t cvt2_f16(float a, float b) {  // packed f16x2 (a in the low half), saturating
    uint32_t d;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;\n" : "=r"(d) : "f"(b), "f"(a));
    return d;
}
// running maximum of |x| over packed f16 pairs (both halves at once): what the fp16 aggregation operand saturates at is detected here
__device__ __forceinline__ uint32_t hmax2_abs(uint32_t acc, uint32_t v) {
    uint32_t a, d;
    asm("abs.f16x2 %0, %1;\n" : "=r"(a) : "r"(v));
    asm("max.f16x2 %0, %1, %2;\n" : "=r"(d) : "r"(acc), "r"(a));
    return d;
}
__device__ __forceinline__ unsigned short f16_bits(float x) { return (unsigned short)(cvt2_f16(x, 0.f) & 0xFFFFu); }
__device__ __forceinline__ float f16_value(unsigned short h) {
    float f;
    asm("cvt.f32.f16 %0, %1;\n" : "=f"(f) : "h"(h));
    return f;
}
// (1 + popcount(open directions))^-1/2 without branches
__device__ __forceinline__ float dinv_sel(int open_mask) {
    const int deg = 1 + __popc(open_mask & 15);
    float d = 1.0f;
    d = deg == 2 ? 0.70710678118654752f : d;
    d = deg == 3 ? 0.57735026918962576f : d;
    d = deg == 4 ? 0.5f : d;
    d = deg == 5 ? 0.44721359549995794f : d;
    return d;
}
// one lane of a fully converged warp
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}\n" : "=r"(pred));
    return pred != 0;
}
// mbarrier wait: hint_ns == 0 spins on try_wait, otherwise passes the suspend-time hint
__device__ __forceinline__ void mbar_wait2(uint32_t bar, uint32_t parity, uint32_t hint_ns) {
    uint32_t ok = 0;
    if (hint_ns == 0) {
        while (!ok)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                         : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } else {
        while (!ok)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                         : "=r"(ok) : "r"(bar), "r"(parity), "r"(hint_ns) : "memory");
    }
}
__device__ __forceinline__ void sts128(uint32_t saddr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts16(uint32_t saddr, unsigned short v) {
    asm volatile("st.shared.b16 [%0], %1;\n" ::"r"(saddr), "h"(v) : "memory");
}

// Accumulator columns [32 cb, 32 cb + 32) of this thread's lane -> bf16 -> node block cb of the thread's feature row.
// Nodes >= 81 are written as zero (they are K padding of the aggregation's A operand: 0 x garbage must not be NaN).
// (Tried and dropped: converting every other relu -> bf16 pair on the FMA pipe with a Veltkamp split -- 9 full-rate instructions
// per pair against one F2FP at 16 cycles per warp instruction -- made the kernel 9 % slower: issue slots and registers.)
enum { kToBf16 = 0, kToBf16Relu = 1, kToF16 = 2 };
template <int kMode>
__device__ __forceinline__ uint32_t cvt_pair(float a, float b) {
    return kMode == kToF16 ? cvt2_f16(a, b) : cvt2<kMode == kToBf16Relu>(a, b);
}
// grow != nullptr (training forward): the same 16-byte chunks also go to the board's saved tile in global memory.
// kToF16: `amax` (packed f16x2) collects the largest |z| of the thread's row, so that a saturated conversion is noticed.
template <int kMode>
__device__ __forceinline__ void store_block(uint32_t row_addr, int swz, int cb, const float *z, unsigned char *grow, uint32_t &amax) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        uint4 v;
        if (cb == 2 && q == 3) v = make_uint4(0u, 0u, 0u, 0u);                                   // nodes 88..95
        else if (cb == 2 && q == 2) v = make_uint4(cvt_pair<kMode>(z[16], 0.f), 0u, 0u, 0u);     // node 80, then padding
        else {
            v.x = cvt_pair<kMode>(z[q * 8 + 0], z[q * 8 + 1]); v.y = cvt_pair<kMode>(z[q * 8 + 2], z[q * 8 + 3]);
            v.z = cvt_pair<kMode>(z[q * 8 + 4], z[q * 8 + 5]); v.w = cvt_pair<kMode>(z[q * 8 + 6], z[q * 8 + 7]);
        }
        if (kMode == kToF16) {
            amax = hmax2_abs(amax, v.x);
            if (!(cb == 2 && q == 2)) amax = hmax2_abs(hmax2_abs(hmax2_abs(amax, v.y), v.z), v.w);
        }
        sts128(row_addr + (uint32_t)cb * kFmBlock + (uint32_t)((q ^ swz) << 4), v);
        if (grow) *reinterpret_cast<uint4 *>(grow + (uint32_t)cb * kFmBlock + (uint32_t)((q ^ swz) << 4)) = v;
    }
}

// the three column blocks of this thread's accumulator lane (+ bias) -> its feature row
template <int kMode>
__device__ __forceinline__ void epilogue_store(uint32_t tmem_me, uint32_t row_addr, int swz, float bias, uint32_t &amax, unsigned char *grow = nullptr) {
#pragma unroll
    for (int cb = 0; cb < 3; ++cb) {
        float z[32];
        tmem_ld32(tmem_me + cb * 32, z);
        if (bias != 0.f) {   // (0 where the bias is already inside the MMA or not wanted)
#pragma unroll
            for (int i = 0; i < 32; ++i) z[i] += bias;
        }
        store_block<kMode>(row_addr, swz, cb, z, grow, amax);
    }
}

// kSave (training forward, precision 1): additionally writes what gcn_backward_tc2_kernel needs (layout: gnn_layout.cuh, Tc2Saved):
// the X1^T and X2^T tiles byte for byte as they sit in shared memory, the ReLU mask of layer 3 (81 bits per feature), the
// layer-1 node operand transposed [16][96] as a K-major SWIZZLE_64B tile, and the A_hat coefficients rounded to tf32.
// kLegal (inference of a leaf evaluation): 640 threads, the fifth warpgroup writes the legal mask and pawn moves (legal_warpgroup).
// Registers: launched at 96 per thread; the legal warpgroup gives up 32 (setmaxnreg.dec to 64), the trunk groups take 8 more
// (setmaxnreg.inc to 104): 512 x 104 + 128 x 64 = 640 x 96.
template <bool kSave, bool kLegal>
__global__ void __launch_bounds__(kTrunkThreads + (kLegal ? kLegalThreads : 0), 1)
gcn_forward_tc2_kernel(const float *__restrict__ params, const unsigned char *__restrict__ prepared,
                       const AqState *__restrict__ states, int64_t B, float *__restrict__ pooled_out, float *__restrict__ saved,
                       uint32_t wait_ns, uint32_t *mask, uint8_t *pawn) {
    extern __shared__ unsigned char smem_raw[];
    Tc2Smem &sm = *reinterpret_cast<Tc2Smem *>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int gtid = threadIdx.x;
#if TC2_FINISH
    const long long clk0 = clock64();
    if (gtid == 0 && blockIdx.x < kFinishCtas) g_tc2_finish[blockIdx.x][0] = globaltimer_ns();
#endif
    const int grp = gtid / kGroupThreads, tid = gtid % kGroupThreads;  // tid = feature = TMEM lane
    Tc2Group &gs = sm.g[grp];

    // the next kernel in the stream (the heads) may be launched now: it loads its weight tiles while this grid drains and waits for
    // this grid's completion (griddepcontrol.wait) before it reads the pooled activations
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    if constexpr (kLegal) {
        if (gtid >= kTrunkThreads) {  // warp-uniform: the legal warpgroup never touches tensor memory nor a trunk barrier
            asm volatile("setmaxnreg.dec.sync.aligned.u32 64;\n" ::: "memory");
            legal_warpgroup(states, B, mask, pawn, *reinterpret_cast<Tc2Legal *>(reinterpret_cast<unsigned char *>(&sm) + sizeof(Tc2Smem)),
                            gtid - kTrunkThreads);
#if TC2_FINISH
            if (gtid == kTrunkThreads && blockIdx.x < kFinishCtas) {
                g_tc2_finish[blockIdx.x][1] = globaltimer_ns();
                g_tc2_finish[blockIdx.x][3] = (unsigned long long)(clock64() - clk0);
            }
#endif
            return;
        }
        asm volatile("setmaxnreg.inc.sync.aligned.u32 104;\n" ::: "memory");
    }
    // ---- one-time setup ---------------------------------------------------------------------------------------
    {
        uint4 *adj = reinterpret_cast<uint4 *>(&gs.adj[0][0][0]);  // adjacency tiles start as zero; only the stencil positions change
        for (int c = tid; c < (int)(4 * kAdjBlock / 16); c += kGroupThreads) adj[c] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (gtid < kV) {
        const int v = gtid, r = v / 9, c = v - 9 * r;
        NodeConst k;
        const uint32_t none = 0x80000000u;
        k.upm = r >= 1 ? ((c >= 1 ? 1u : 0u) | (c <= 7 ? 2u : 0u)) : none;                 // H slots (r-1, c-1), (r-1, c)
        k.dnm = r <= 7 ? ((c >= 1 ? 1u << 8 : 0u) | (c <= 7 ? 1u << 9 : 0u)) : none;       // H slots (r, c-1), (r, c)
        k.lfm = c >= 1 ? ((r >= 1 ? 1u : 0u) | (r <= 7 ? 1u << 8 : 0u)) : none;            // V slots (r-1, c-1), (r, c-1)
        k.rtm = c <= 7 ? ((r >= 1 ? 2u : 0u) | (r <= 7 ? 1u << 9 : 0u)) : none;            // V slots (r-1, c), (r, c)
        k.pv = ((r <= 7 && c <= 7) ? 1u << 9 : 0u) | ((r >= 1 && c <= 7) ? 2u : 0u) | ((r <= 6 && c <= 7) ? 1u << 17 : 0u) |
               ((r <= 7 && c >= 1) ? 1u << 8 : 0u) | ((r <= 7 && c <= 6) ? 1u << 10 : 0u);
        k.sh = (uint32_t)(8 * r + c);
        const int blk = v >= 48 ? 1 : 0, row = v - 48 * blk, kl0 = v - 32 * blk;  // row and self position inside the block's window
        auto off = [&](int kl, bool exists) -> uint32_t {
            return exists ? (uint32_t)blk * kAdjBlock + (uint32_t)row * 128u + (uint32_t)(((kl >> 3) ^ (row & 7)) << 4) + (uint32_t)(kl & 7) * 2u
                          : 0xFFFFu;
        };
        k.adj01 = off(kl0, true) | (off(kl0 - 9, r >= 1) << 16);
        k.adj23 = off(kl0 + 9, r <= 7) | (off(kl0 - 1, c >= 1) << 16);
        k.adj4 = off(kl0 + 1, c <= 7);
        k.row_off = sw32_chunk(v, 0);  // chunk 0 of row v in the K-major SWIZZLE_32B layer-1 operand; chunk 1 = ^ 16
        k.pad0 = k.pad1 = 0u;
        sm.nc[v] = k;
    } else if (gtid >= 128 && gtid < 192) {
        const int i = gtid - 128, a = i >> 3, b2 = i & 7;
        float cf = 0.f;
        if (a >= 1 && a <= 5 && b2 >= 1 && b2 <= 5) cf = dinv_sel((1 << (a - 1)) - 1) * dinv_sel((1 << (b2 - 1)) - 1);  // popcount(2^k - 1) = k
        sm.lut[i] = make_float2(cf, __uint_as_float((uint32_t)f16_bits(cf)));
    }
    if (tid < 32) reinterpret_cast<uint32_t *>(gs.deg)[tid] = 0x01010101u;
    if (gtid < kH) {
        const int n = gtid;
        uint4 c0, c1;
        if (prepared) {  // layer-1 operand as built by aq_prepare_inference
            c0 = __ldg(reinterpret_cast<const uint4 *>(prepared + kPrepW1 + sw32_chunk(n, 0)));
            c1 = __ldg(reinterpret_cast<const uint4 *>(prepared + kPrepW1 + sw32_chunk(n, 1)));
        } else {
            float w[kF];
#pragma unroll
            for (int f = 0; f < kF; ++f) w[f] = __ldg(params + kOffW1 + n * kF + f);
            const float bias = __ldg(params + kOffB1 + n);
            const float bias_hi = __bfloat162float(__float2bfloat16_rn(bias));
            c0.x = pack_bf16(w[0], w[1]); c0.y = pack_bf16(w[2], w[3]); c0.z = pack_bf16(w[4], w[5]); c0.w = pack_bf16(w[0], w[1]);
            c1.x = pack_bf16(w[2], w[3]); c1.y = pack_bf16(w[4], w[5]); c1.z = pack_bf16(bias_hi, bias - bias_hi); c1.w = 0u;
        }
        *reinterpret_cast<uint4 *>(sm.w1 + sw32_chunk(n, 0)) = c0;
        *reinterpret_cast<uint4 *>(sm.w1 + sw32_chunk(n, 1)) = c1;
    }
    if (gtid < kG) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(smem_u32(&sm.mbar[gtid])) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (gtid < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&sm.tmem_base)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    if constexpr (kLegal) trunk_sync(); else __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = sm.tmem_base;
    const uint32_t lane_off = (uint32_t)((tid >> 5) * 32) << 16;  // this warp's TMEM lane quadrant
    constexpr int kWeightGroups = 2;   // W2 (group 0) / W3 (group 1)
    if (grp < kWeightGroups) {  // row `tid` -> 64 TMEM columns, two bf16 per column (k = 2c, 2c + 1)
        const bool w3 = grp != 0;
        const uint32_t dst = tmem_base + lane_off + (w3 ? kTmemW3 : kTmemW2);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            uint32_t r[32];
            if (prepared) {
                const unsigned char *src = prepared + (w3 ? kPrepW3 : kPrepW2);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(src + sw128_chunk(tid, half * 8 + j, kWKBlock)));
                    r[4 * j] = v.x; r[4 * j + 1] = v.y; r[4 * j + 2] = v.z; r[4 * j + 3] = v.w;
                }
            } else {
                const float4 *W = reinterpret_cast<const float4 *>(params + (w3 ? kOffW3 : kOffW2) + tid * kH + half * 64);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float4 v = __ldg(W + j);
                    r[2 * j] = pack_bf16(v.x, v.y); r[2 * j + 1] = pack_bf16(v.z, v.w);
                }
            }
            tmem_st32(dst + half * 32, r);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    if constexpr (kLegal) trunk_sync(); else __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");

    const uint32_t tmem_d = tmem_base + (uint32_t)grp * kGroupCols;    // the group's accumulator columns
    const uint32_t tmem_me = tmem_d + lane_off;
    const uint32_t bar = smem_u32(&sm.mbar[grp]);
    const uint32_t fm_addr = smem_u32(gs.fm), adj_addr = smem_u32(&gs.adj[0][0][0]), l1_addr = smem_u32(gs.l1op);
    const uint32_t w1_addr = smem_u32(sm.w1);
    const uint32_t row_addr = fm_addr + (uint32_t)(tid >> 3) * 512u + (uint32_t)(tid & 7) * 64u;  // this thread's feature row
    const int swz = (tid & 7) >> 1;
    const uint32_t row_off = (uint32_t)(tid >> 3) * 512u + (uint32_t)(tid & 7) * 64u;
    const Tc2Saved SV{B};
    const float bias2 = __ldg(params + kOffB2 + tid), bias3 = __ldg(params + kOffB3 + tid);   // added in the epilogues (fp32)
    uint32_t phase = 0;
    // The MMAs of a group are issued by its first warp from WARP-UNIFORM values (everything below derives from a shuffled warp
    // index), so that descriptors live in uniform registers and one tcgen05.mma costs a few instructions instead of a
    // per-thread register -> uniform register broadcast loop.
    const int warp_u = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int grp_u = warp_u >> 2;
    const bool issuer_warp = (warp_u & 3) == 0;
    const uint32_t tmem_base_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t tmem_d_u = tmem_base_u + (uint32_t)grp_u * kGroupCols;
    const uint32_t smem_u = smem_u32(&sm);
    const uint32_t fm_u = smem_u + (uint32_t)offsetof(Tc2Smem, g) + (uint32_t)grp_u * (uint32_t)sizeof(Tc2Group);
    const uint32_t adj_u = fm_u + (uint32_t)offsetof(Tc2Group, adj), l1_u = fm_u + (uint32_t)offsetof(Tc2Group, l1op);
    const uint32_t w1_u = smem_u + (uint32_t)offsetof(Tc2Smem, w1);
    const uint32_t bar_u = smem_u + (uint32_t)offsetof(Tc2Smem, mbar) + (uint32_t)grp_u * 8u;

    const int64_t stride = (int64_t)gridDim.x * kG;
#if TC2_PREFETCH
    uint4 pre_a = make_uint4(0u, 0u, 0u, 0u);
    uint32_t pre_b = 0u;
    if ((int64_t)blockIdx.x * kG + grp < B && tid < kV) {
        pre_a = __ldg(reinterpret_cast<const uint4 *>(states + (int64_t)blockIdx.x * kG + grp));
        pre_b = __ldg(reinterpret_cast<const uint32_t *>(states + (int64_t)blockIdx.x * kG + grp) + 4);
    }
#endif
#if TC2_TIMING
    long long t_last = clock64();
#endif
    // Node phase of board bn: fills the adjacency tile at adj_dst and the layer-1 node operand.  It contains one group barrier
    // (all 128 threads of the group call it).
    auto node_phase = [&](int64_t bn, uint32_t adj_dst) {
        // ---- node threads, part 1: open directions of node v from two bitboard windows; degree -> shared memory ----------
        uint32_t wH = 0u, wV = 0u, meta = 0u;
        int m = 0, dv = 1;
        if (tid < kV) {
#if TC2_PREFETCH
            const u64 h = ((u64)pre_a.y << 32) | pre_a.x, vw = ((u64)pre_a.w << 32) | pre_a.z;
            meta = pre_b;
            if (bn + stride < B) {
                pre_a = __ldg(reinterpret_cast<const uint4 *>(states + bn + stride));
                pre_b = __ldg(reinterpret_cast<const uint32_t *>(states + bn + stride) + 4);
            }
#else
            const uint4 sa = __ldg(reinterpret_cast<const uint4 *>(states + bn));
            meta = __ldg(reinterpret_cast<const uint32_t *>(states + bn) + 4);
            const u64 h = ((u64)sa.y << 32) | sa.x, vw = ((u64)sa.w << 32) | sa.z;
#endif
            const uint4 k0 = *reinterpret_cast<const uint4 *>(&sm.nc[tid].upm);
            const uint32_t sh = sm.nc[tid].sh;
            wH = (uint32_t)((((unsigned __int128)h) << 9) >> sh);
            wV = (uint32_t)((((unsigned __int128)vw) << 9) >> sh);
            const uint32_t eH = wH | 0x80000000u, eV = wV | 0x80000000u;
            m = ((eH & k0.x) == 0u ? 1 : 0) | ((eH & k0.y) == 0u ? 2 : 0) | ((eV & k0.z) == 0u ? 4 : 0) | ((eV & k0.w) == 0u ? 8 : 0);
            dv = 1 + __popc(m);
            gs.deg[16 + tid] = (uint8_t)dv;
        }
        group_sync(grp);
        // ---- part 2: A_hat row of v -> adjacency tile (fp16 bits straight from a table), and the layer-1 node operand row
        //      [hi(A_hat x0) (6) | lo(A_hat x0) (6) | 1 | 1 | 0 | 0]; the six planes of pieces_array (game_logic.py:56-93) at v and
        //      its neighbours are read from the same windows -------------------------------------------------------------------
        if (tid < kV) {
            const int v = tid;
            const uint4 k1 = *reinterpret_cast<const uint4 *>(&sm.nc[tid].pv);
            const uint2 k2 = *reinterpret_cast<const uint2 *>(&sm.nc[tid].adj4);
            const int du = gs.deg[16 + v - 9], dd = gs.deg[16 + v + 9], dl = gs.deg[16 + v - 1], dr = gs.deg[16 + v + 1];
            const float2 e0 = sm.lut[dv * 9];
            const float2 eu = sm.lut[(m & 1) ? dv * 8 + du : 0], ed = sm.lut[(m & 2) ? dv * 8 + dd : 0];
            const float2 el = sm.lut[(m & 4) ? dv * 8 + dl : 0], er = sm.lut[(m & 8) ? dv * 8 + dr : 0];
            const float c0 = e0.x, cu = eu.x, cd = ed.x, cl = el.x, cr = er.x;
            {
                const uint32_t o0 = k1.z & 0xFFFFu, o1 = k1.z >> 16, o2 = k1.w & 0xFFFFu, o3 = k1.w >> 16, o4 = k2.x;
                sts16(adj_dst + o0, (unsigned short)__float_as_uint(e0.y));
                if (o1 != 0xFFFFu) sts16(adj_dst + o1, (unsigned short)__float_as_uint(eu.y));
                if (o2 != 0xFFFFu) sts16(adj_dst + o2, (unsigned short)__float_as_uint(ed.y));
                if (o3 != 0xFFFFu) sts16(adj_dst + o3, (unsigned short)__float_as_uint(el.y));
                if (o4 != 0xFFFFu) sts16(adj_dst + o4, (unsigned short)__float_as_uint(er.y));
            }
            float s[kF];
            {
                const int dp = (int)(meta & 0xFF) - v, de = (int)((meta >> 16) & 0xFF) - v;
                const float pw = (float)((meta >> 8) & 0xFF), ew = (float)(meta >> 24);
                const uint32_t pH = wH & k1.x, pV = wV & k1.x;
                auto onehot = [&](int d) {  // same summation order as a fused multiply-add chain over {self, up, down, left, right}
                    float t = d == 0 ? c0 : 0.f;
                    t += d == -9 ? cu : 0.f; t += d == 9 ? cd : 0.f; t += d == -1 ? cl : 0.f; t += d == 1 ? cr : 0.f;
                    return t;
                };
                auto plane = [&](uint32_t w) {
                    float t = (w & (1u << 9)) ? c0 : 0.f;
                    t += (w & 2u) ? cu : 0.f; t += (w & (1u << 17)) ? cd : 0.f; t += (w & (1u << 8)) ? cl : 0.f; t += (w & (1u << 10)) ? cr : 0.f;
                    return t;
                };
                auto scaled = [&](float x) { return fmaf(cr, x, fmaf(cl, x, fmaf(cd, x, fmaf(cu, x, c0 * x)))); };
                s[0] = onehot(dp); s[1] = scaled(pw); s[2] = onehot(de); s[3] = scaled(ew); s[4] = plane(pH); s[5] = plane(pV);
            }
            uint4 c0v, c1v;
            c0v.x = cvt2<false>(s[0], s[1]); c0v.y = cvt2<false>(s[2], s[3]); c0v.z = cvt2<false>(s[4], s[5]);
            c0v.w = cvt2<false>(s[0] - __uint_as_float(c0v.x << 16), s[1] - __uint_as_float(c0v.x & 0xFFFF0000u));
            c1v.x = cvt2<false>(s[2] - __uint_as_float(c0v.y << 16), s[3] - __uint_as_float(c0v.y & 0xFFFF0000u));
            c1v.y = cvt2<false>(s[4] - __uint_as_float(c0v.z << 16), s[5] - __uint_as_float(c0v.z & 0xFFFF0000u));
            c1v.z = 0x3F803F80u; c1v.w = 0u;  // 1, 1, 0, 0
            sts128(l1_addr + k2.y, c0v);
            sts128(l1_addr + (k2.y ^ 16u), c1v);
            if (kSave) {
                auto tf = [](float c) { return __uint_as_float((__float_as_uint(c) + 0x1000u) & 0xFFFFE000u); };
                float4 *cf = reinterpret_cast<float4 *>(SV.coef(saved, bn) + v * 8);
                cf[0] = make_float4(tf(c0), tf(cu), tf(cd), tf(cl));
                cf[1] = make_float4(tf(cr), 0.f, 0.f, 0.f);
                unsigned char *at = SV.a1t(saved, bn);
                const uint32_t wds[8] = {c0v.x, c0v.y, c0v.z, c0v.w, c1v.x, c1v.y, c1v.z, c1v.w};
#pragma unroll
                for (int k = 0; k < 16; ++k)
                    *reinterpret_cast<unsigned short *>(at + Tc2Saved::a1t_off(k, v)) = (unsigned short)(wds[k >> 1] >> (16 * (k & 1)));
            }
        } else if (kSave && tid < kNodesPad) {  // node padding of the transposed layer-1 operand must be zero (it is K of dW1)
            unsigned char *at = SV.a1t(saved, bn);
#pragma unroll
            for (int k = 0; k < 16; ++k) *reinterpret_cast<unsigned short *>(at + Tc2Saved::a1t_off(k, tid)) = 0;
        }
    };
    uint32_t par = 0;  // adjacency buffer of the current board
    {
        const int64_t b0 = (int64_t)blockIdx.x * kG + grp;
        if (b0 < B) node_phase(b0, adj_addr);
    }
    for (int64_t b = (int64_t)blockIdx.x * kG + grp; b < B; b += stride) {
        TC2_T(2);
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
        group_sync(grp);
        TC2_T(3);
        if (issuer_warp) {
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            if (elect_one()) {
                mma_bf16(tmem_d_u, desc_sw32(w1_u), desc_sw32(l1_u), kIdescL1, 0u);  // one K = 16 step
                mma_commit(bar_u);
            }
            __syncwarp();
        }
        mbar_wait2(bar, phase, wait_ns);
        phase ^= 1u;
        TC2_T(4);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        // ---- layer 1 epilogue: ReLU -> bf16 -> X1^T row ---------------------------------------------------------------
        uint32_t amax = 0u;  // largest |Z| (packed f16x2) this thread converted for this board
        epilogue_store<kToBf16Relu>(tmem_me, row_addr, swz, 0.f, amax);   // (b1 is folded into the layer-1 MMA)
        float pool = 0.f;
#pragma unroll 1
        for (int layer = 1; layer < kLayers; ++layer) {
            // ---- transform: Z^T = W X^T (A = W in TMEM, B = X^T tile) -------------------------------------------
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
            group_sync(grp);
        TC2_T(5);
            if (issuer_warp) {
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                if (elect_one()) {
                    const uint32_t w_tmem = tmem_base_u + (layer == 1 ? kTmemW2 : kTmemW3);
                    if (kSave) {  // training forward: the X^T tile just completed goes to global memory as one bulk copy (TMA), byte for byte
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n"
                                     ::"l"(SV.xt(saved, layer - 1, b)), "r"(fm_u), "r"(3u * kFmBlock) : "memory");
                        asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
                    }
                    {
#pragma unroll
                        for (int k = 0; k < 8; ++k)  // K = 128 features = 8 x 16: 8 TMEM columns of A, two 8-feature atoms of B per step
                            mma_ts(tmem_d_u, w_tmem + k * 8, desc_fm_mn(fm_u + k * 1024), kIdescT, k > 0 ? 1u : 0u);
                    }
                    // the tile is overwritten after this phase: the commit is held back until the bulk copy has read it
                    if (kSave) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
                    mma_commit(bar_u);
                }
                __syncwarp();
            }
            mbar_wait2(bar, phase, wait_ns);
            phase ^= 1u;
        TC2_T(6);
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            // ---- Z^T -> fp16 -> the same tile, now the aggregation's A operand -------------------------------------
            epilogue_store<kToF16>(tmem_me, row_addr, swz, 0.f, amax);
            // ---- aggregate: Y^T = Z^T A_hat^T + b 1^T --------------------------------------------------------------
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
            group_sync(grp);
        TC2_T(7);
            {
                const uint32_t par_u = __shfl_sync(0xffffffffu, par, 0);
                if (issuer_warp) {
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    if (elect_one()) {
#pragma unroll
                        for (int blk = 0; blk < 2; ++blk) {
                            const uint32_t d = tmem_d_u + blk * 48;
#pragma unroll
                            for (int s = 0; s < 4; ++s) {  // 64 in-nodes = 4 K steps; A: two 32-node blocks, 2 steps of 32 B each
                                const uint64_t bd = desc_sw128(adj_u + (par_u * 2u + (uint32_t)blk) * kAdjBlock + (uint32_t)s * 32u);
                                const uint64_t a = desc_fm_k(fm_u + (uint32_t)(blk + (s >> 1)) * kFmBlock + (uint32_t)(s & 1) * 32u);
                                mma_bf16(d, a, bd, kIdescA, s ? 1u : 0u);
                            }
                        }
                        mma_commit(bar_u);
                    }
                    __syncwarp();
                }
            }
            // while the last aggregation runs: the node phase of this group's next board (other adjacency buffer)
            if (layer + 1 == kLayers && b + stride < B) node_phase(b + stride, adj_addr + (par ^ 1u) * 2u * kAdjBlock);
            mbar_wait2(bar, phase, wait_ns);
            phase ^= 1u;
        TC2_T(8);
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            if (layer + 1 < kLayers) {  // + bias -> ReLU -> bf16 -> X^T row of the next layer
                epilogue_store<kToBf16Relu>(tmem_me, row_addr, swz, bias2, amax);
            } else {                    // last layer feeds only the mean pool
#pragma unroll
                uint32_t m3[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                for (int cb = 0; cb < 3; ++cb) {
                    float z[32];
                    tmem_ld32(tmem_me + cb * 32, z);
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (cb * 32 + i < kV) {
                            const float y = z[i] + bias3;
                            pool += fmaxf(y, 0.f);
                            if (kSave) m3[cb] |= (y > 0.f ? 1u : 0u) << i;
                        }
                }
                if (kSave) *reinterpret_cast<uint4 *>(SV.mask3(saved, b) + tid * 16) = make_uint4(m3[0], m3[1], m3[2], 0u);
            }
        }
        // The aggregation operand is fp16: a transform output beyond +-65504 would be clamped by the saturating conversion.  That is
        // never passed on silently: the feature's pooled value becomes NaN, so the board's policy and value come out as NaN
        // (fp32 precision has no such limit; DESIGN.md section 8).
        const bool clamped = (amax & 0x7FFFu) >= 0x7BFFu || (amax >> 16) >= 0x7BFFu;
        pooled_out[b * kH + tid] = clamped ? __int_as_float(0x7FC00000) : pool / (float)kV;
        par ^= 1u;
        TC2_T(9);
        // no barrier here: the next board's first MMA is issued behind a group barrier that every thread reaches after its pool loads
        TC2_T(10);
    }
    // ---- teardown ---------------------------------------------------------------------------------------------------
#if TC2_FINISH
    if (tid == 0 && blockIdx.x < kFinishCtas) {
        atomicMax(&g_tc2_finish[blockIdx.x][2], globaltimer_ns());
        atomicMax(&g_tc2_finish[blockIdx.x][4], (unsigned long long)(clock64() - clk0));
        if (grp == 0) g_tc2_finish[blockIdx.x][5] = (unsigned long long)((B - (int64_t)blockIdx.x * kG + stride - 1) / stride);
    }
#endif
    if (!kLegal) aq_pdl_wait();  // programmatic launch behind the legal-mask kernels: this grid is complete only once they are (no-op otherwise)
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    if constexpr (kLegal) trunk_sync(); else __syncthreads();
    if (gtid < 32) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

}  // namespace

// Trunk, version 2.  saved == nullptr: inference (same contract as aq_gcn_forward_tc); saved != nullptr: training forward, precision 1,
// activations kept in the Tc2Saved layout for aq_gcn_backward_tc2.
// mask != nullptr (inference only): the leaf evaluation's legal mask [B][8] and pawn moves [B][8] are computed by the same launch, in a
// fifth warpgroup of every CTA that runs beside the trunk groups (the trunk does not read them; the heads kernel behind it does).
// after_legal (inference without mask): the predecessor in the stream is the legal-mask kernel of the same leaf evaluation, whose
// output this kernel does not read: the grid is launched programmatically (it starts on SMs as the legal-mask grid drains from them)
// and orders itself behind that grid only at its very end (aq_pdl_wait before the teardown), so that the heads kernel behind it sees
// the mask.
int aq_gcn_forward_tc2(const float *params, const void *prepared, const AqState *states, int64_t B, float *pooled, float *saved,
                       uint32_t *mask, uint8_t *pawn, bool after_legal, cudaStream_t st) {
    static int sms = 0;
    const uint32_t wait_ns = 0;  // suspend-time hint of the mbarrier waits (0 = spin; measured best)
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    const size_t smem = sizeof(Tc2Smem) + 1024;
    const int64_t want = (B + kG - 1) / kG;
    const unsigned grid = (unsigned)(want < sms ? want : sms);
    const unsigned char *prep = reinterpret_cast<const unsigned char *>(prepared);
    cudaError_t e;
    if (saved) {
        e = cudaFuncSetAttribute(gcn_forward_tc2_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return aq_set_error((int)e, "gcn_forward_tc2 smem");
        gcn_forward_tc2_kernel<true, false><<<grid, kTrunkThreads, smem, st>>>(params, prep, states, B, pooled, saved, wait_ns, nullptr, nullptr);
    } else if (mask) {
        const size_t smem_l = smem + sizeof(Tc2Legal);
        e = cudaFuncSetAttribute(gcn_forward_tc2_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_l);
        if (e != cudaSuccess) return aq_set_error((int)e, "gcn_forward_tc2 smem");
        gcn_forward_tc2_kernel<false, true><<<grid, kTrunkThreads + kLegalThreads, smem_l, st>>>(params, prep, states, B, pooled, nullptr, wait_ns,
                                                                                                 mask, pawn);
    } else {
        e = cudaFuncSetAttribute(gcn_forward_tc2_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return aq_set_error((int)e, "gcn_forward_tc2 smem");
        if (after_legal) {
            e = aq_launch_pdl(gcn_forward_tc2_kernel<false, false>, dim3(grid), dim3(kTrunkThreads), smem, st, params, prep, states, B, pooled,
                              (float *)nullptr, wait_ns, (uint32_t *)nullptr, (uint8_t *)nullptr);
            if (e != cudaSuccess) return aq_set_error((int)e, "gcn_forward_tc2_kernel(launch)");
        } else {
            gcn_forward_tc2_kernel<false, false><<<grid, kTrunkThreads, smem, st>>>(params, prep, states, B, pooled, nullptr, wait_ns, nullptr,
                                                                                    nullptr);
        }
    }
    return aq_check_launch("gcn_forward_tc2_kernel");
}
