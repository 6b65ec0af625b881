// Tensor-core backward of the GCN trunk, version 2 -- the counterpart of gcn_forward_tc2_kernel<kSave = true> (gnn_tc2.cu).
// As in the forward, every product is feature-major (one FEATURE per TMEM lane, the board's nodes along the columns) and the
// aggregation of the gradient runs on the tensor cores too; no stencil arithmetic, no node-major scattered stores.
//
// One CTA per SM, persistent over boards: 256 threads = two threads per TMEM lane (feature); the thread with half index h owns node
// columns [48 h, 48 h + 48) of every accumulator row it touches, so each epilogue phase of the (single) dependency chain is split
// in two.  Per board and layer l = 3, 2:
//     dY_l = (X_l > 0) * dX_l          thread f masks its lane of the dX accumulator IN PLACE (tcgen05.ld / tcgen05.st)   (dX_3 = dg / 81)
//     dZ_l^T = dY_l^T A_hat^T          kind::tf32  A = dY_l^T, the fp32 accumulator columns read in place (A_hat is symmetric: the
//                                                  transposed-CSR scatter of the backward is the same gather), B = A_hat (tf32, banded)
//     dZ_l^T -> bf16 -> feature-major tile (thread f writes its own row, 16-byte stores)
//     dX_{l-1}^T = W_l^T dZ_l^T        kind::f16   A = W_l^T [k][n] (shared memory), B = the tile read MN-major [K = n][N = nodes]
//     dW_l      += dZ_l^T X_{l-1}      kind::f16   A = the same tile read K-major [M = n][K = nodes], B = X_{l-1}^T tile saved by the forward
// and for layer 1 (forward: Y_1 = (A_hat X0 | 1) W1ext^T):  dW1ext += dY_1^T A1  with A1^T saved as a [16][96] tile.
// TF32 keeps the gradient's fp32 exponent range (an fp16 aggregation would underflow: dg / 81 / batch is ~1e-7).
// The weight-gradient accumulators live in TMEM for the whole kernel (accumulate across boards) and are written once per CTA into
// its slot of the partial-gradient buffer; reduce_partials_kernel sums the slots in a fixed order (deterministic, atomic-free).
#include <cstddef>
#include <cuda_bf16.h>
#include "gnn_fp32.cuh"
#include "tc_common.cuh"

using namespace aq;
using namespace aqtc;

#ifndef TC2B_TIMING
#define TC2B_TIMING 0    // 1: per-phase clock64 accounting by thread 0 of CTA 0 (debug variant, scripts/bwd_timing.py)
#endif
#if TC2B_TIMING
__device__ long long g_tc2b_timing[16];
#define TC2B_T(slot) do { if (blockIdx.x == 0 && gtid == 0) { const long long t_ = clock64(); g_tc2b_timing[slot] += t_ - t_last; t_last = t_; } } while (0)
extern "C" int aq_debug_bwd_timing(long long *out) {
    cudaMemcpyFromSymbol(out, g_tc2b_timing, sizeof(long long) * 16);
    long long z[16] = {0};
    cudaMemcpyToSymbol(g_tc2b_timing, z, sizeof(z));
    return 0;
}
#else
#define TC2B_T(slot) do { } while (0)
#endif

namespace {

constexpr int kNodesPad = 96;
constexpr uint32_t kFmBlock = 16 * 512;     // feature-major tile: [3 node blocks of 32][16 atoms of 8 features][8][64 B]
constexpr uint32_t kRowBlock = 128 * 128;   // K-block of a 128-row K-major SWIZZLE_128B tile (W^T)
constexpr uint32_t kAdjKBlock = 48 * 128;   // adjacency block, one K-block: 48 out-node rows x 32 in-nodes (tf32, 128 B)
constexpr uint32_t kAdjBlock = 2 * kAdjKBlock;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColX = 0, kColZ = 96, kColW3 = 192, kColW2 = 320, kColW1 = 448;  // TMEM column map (464 used)

constexpr uint32_t kIdescBase = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24);                  // D = f32, A = B = bf16, M = 128
constexpr uint32_t kIdescDX = kIdescBase | (1u << 16) | ((uint32_t)(kNodesPad >> 3) << 17);                // B MN-major, N = 96
constexpr uint32_t kIdescDW = kIdescBase | ((uint32_t)(128 >> 3) << 17);                                   // K-major, N = 128
constexpr uint32_t kIdescDW1 = kIdescBase | ((uint32_t)(16 >> 3) << 17);                                   // K-major, N = 16
constexpr uint32_t kIdescAgg = (1u << 4) | (2u << 7) | (2u << 10) | ((128u >> 4) << 24) | ((uint32_t)(48 >> 3) << 17);  // tf32, N = 48

struct BoardIn {
    unsigned char xt2[3 * kFmBlock];    // X2^T tile (bf16, feature-major): B operand of dW3, and the ReLU mask of layer 2
    unsigned char xt1[3 * kFmBlock];    // X1^T tile: B operand of dW2, and the ReLU mask of layer 1
    unsigned char a1t[3 * 1024];        // layer-1 node operand transposed [16][96], K-major SWIZZLE_64B: B operand of dW1ext
    float coef[kV * 8 + 120];           // A_hat coefficients [81][8] (tf32): {self, up, down, left, right, 0, 0, 0}
};
static_assert(sizeof(BoardIn) % 1024 == 0, "board inputs must keep 1024-byte alignment");

struct Bwd2Smem {
    unsigned char w2t[2 * kRowBlock];   // W2^T: row k, K = n  (K-major SWIZZLE_128B)
    unsigned char w3t[2 * kRowBlock];
    unsigned char fm[3 * kFmBlock];     // dZ^T (bf16, feature-major)
    unsigned char adj[2 * kAdjBlock];   // A_hat (tf32), two blocks of [48 out nodes][64 in nodes]
    BoardIn in[2];                      // what the forward saved for a board, double-buffered: the next board's arrives (cp.async) during this one
    unsigned long long mbar;            // aggregation / dX MMAs done (the threads need their result)
    unsigned long long mbar_w;          // weight-gradient MMAs done (only their operand buffers must not be overwritten earlier)
    uint32_t tmem_base;
};
static_assert(sizeof(Bwd2Smem) + 1024 <= 227 * 1024, "Bwd2Smem exceeds shared memory");

__device__ __forceinline__ uint32_t chunk_off128(int row, int j, uint32_t kblock) {  // 16-byte chunk j of `row`, K-major SWIZZLE_128B
    return (uint32_t)(j >> 3) * kblock + (uint32_t)row * 128u + (uint32_t)(((j & 7) ^ (row & 7)) << 4);
}
__device__ __forceinline__ uint64_t desc_fm_mn_b(uint32_t saddr) {  // MN-major SWIZZLE_64B: LBO = node-block stride, SBO = 8-feature atom stride
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(kFmBlock >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
__device__ __forceinline__ uint64_t desc_fm_k_b(uint32_t saddr) {   // K-major SWIZZLE_64B: SBO = 512 B (8 rows x 64 B)
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
__device__ __forceinline__ void mma_ts_tf32_b(uint32_t d, uint32_t a_tmem, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n"
                 ::"r"(d), "r"(a_tmem), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_st32_b(uint32_t taddr, const uint32_t *r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
                 "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
                   "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
                   "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
                   "r"(r[30]), "r"(r[31]) : "memory");
}
__device__ __forceinline__ void tmem_st16_b(uint32_t taddr, const uint32_t *r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
                   "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
// 48 accumulator columns of this thread's lane starting at taddr: one x32 and one x16 load, one wait
__device__ __forceinline__ void tmem_ld48_b(uint32_t taddr, float *v) {
    uint32_t r[48];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]),
          "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47])
        : "r"(taddr + 32) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 48; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st48_b(uint32_t taddr, const uint32_t *r) {
    tmem_st32_b(taddr, r);
    tmem_st16_b(taddr + 32, r + 32);
}
__device__ __forceinline__ void mbar_spin_b(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
}
// bit i of the result = element i of the 8 packed bf16 is > 0 (post-ReLU values are >= 0)
__device__ __forceinline__ uint32_t positive_bits_b(uint4 c) {
    const uint32_t w[4] = {c.x, c.y, c.z, c.w};
    uint32_t m = 0u;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        m |= ((w[i] & 0x7FFFu) != 0u ? 1u : 0u) << (2 * i);
        m |= ((w[i] & 0x7FFF0000u) != 0u ? 1u : 0u) << (2 * i + 1);
    }
    return m;
}

constexpr int kBwdThreads = 256;

__global__ void __launch_bounds__(kBwdThreads, 1)
gcn_backward_tc2_kernel(const float *__restrict__ params, float *__restrict__ saved, const float *dg,
                        int64_t B, float *__restrict__ partial) {
    extern __shared__ unsigned char smem_raw[];
    Bwd2Smem &sm = *reinterpret_cast<Bwd2Smem *>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int gtid = threadIdx.x;
    aq_pdl_trigger();             // the weight-gradient kernel behind this one may be scheduled as SMs free up
    const int tid = gtid & 127;   // = feature = TMEM lane
    const int half = gtid >> 7;   // this thread's node columns: [48 half, 48 half + 48)
    float *slot = partial + (int64_t)blockIdx.x * kNumParams;

    if ((int64_t)blockIdx.x >= B) {  // no board for this CTA: its slot contributes zeros to the GCN ranges
        aq_pdl_wait();               // (the slot may still be read by work queued earlier in the stream)
        for (int i = gtid; i < kOffWP0; i += kBwdThreads) slot[i] = 0.f;
        return;
    }
    // W_l^T tiles: element (row k, col n) = W_l[n][k].  Thread t converts 8 consecutive k of one row n per step (two 16-byte loads,
    // 16 steps in flight) and scatters them into 8 tile rows; a scalar load per iteration serialised 256 L2 round trips per thread.
#pragma unroll 4
    for (int i = gtid; i < 2 * kH * kH / 8; i += kBwdThreads) {
        const int which = i >> 11, e = i & 2047;
        const int n = e >> 4, k0 = (e & 15) * 8;  // coalesced along k
        const float4 lo = __ldg(reinterpret_cast<const float4 *>(params + (which ? kOffW3 : kOffW2) + n * kH + k0));
        const float4 hi = __ldg(reinterpret_cast<const float4 *>(params + (which ? kOffW3 : kOffW2) + n * kH + k0) + 1);
        const float w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
        unsigned char *tile = which ? sm.w3t : sm.w2t;
#pragma unroll
        for (int j = 0; j < 8; ++j)
            *reinterpret_cast<unsigned short *>(tile + chunk_off128(k0 + j, n >> 3, kRowBlock) + (n & 7) * 2) = bf16_bits(w[j]);
    }
    for (int c = gtid; c < (int)(2 * kAdjBlock / 16); c += kBwdThreads)  // adjacency tile starts as zero; only stencil positions change
        reinterpret_cast<uint4 *>(sm.adj)[c] = make_uint4(0u, 0u, 0u, 0u);
    const uint32_t bar = smem_u32(&sm.mbar);
    if (gtid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(bar) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(smem_u32(&sm.mbar_w)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (gtid < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&sm.tmem_base)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");

    const uint32_t tmem = sm.tmem_base;
    const uint32_t lane_base = tmem + ((uint32_t)((tid >> 5) * 32) << 16);   // lane quadrant of this warp (warps w and w + 4 share one)
    const uint32_t col0 = (uint32_t)half * 48u;                              // first of this thread's 48 columns
    const uint32_t w2t_addr = smem_u32(sm.w2t), w3t_addr = smem_u32(sm.w3t), fm_addr = smem_u32(sm.fm);
    const uint32_t adj_addr = smem_u32(sm.adj), in_addr = smem_u32(&sm.in[0]);
    const uint32_t row_off = (uint32_t)(tid >> 3) * 512u + (uint32_t)(tid & 7) * 64u;   // this thread's feature row inside a feature-major tile
    const int swz = (tid & 7) >> 1;
    const bool issuer_warp = __shfl_sync(0xffffffffu, gtid >> 5, 0) == 0;
    // static tile offsets of the 5 stencil positions of node `tid` (self, up, down, left, right); 0xFFFFFFFF = absent
    uint32_t aoff[5] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
    if (gtid < kV) {
        const int v = gtid, r = v / 9, c = v - 9 * r;
        const int blk = v >= 48 ? 1 : 0, row = v - 48 * blk, kl0 = v - 32 * blk;
        auto off = [&](int kl) -> uint32_t {
            return (uint32_t)blk * kAdjBlock + (uint32_t)(kl >> 5) * kAdjKBlock + (uint32_t)row * 128u +
                   (uint32_t)((((kl & 31) >> 2) ^ (row & 7)) << 4) + (uint32_t)(kl & 3) * 4u;
        };
        aoff[0] = off(kl0);
        if (r >= 1) aoff[1] = off(kl0 - 9);
        if (r <= 7) aoff[2] = off(kl0 + 9);
        if (c >= 1) aoff[3] = off(kl0 - 1);
        if (c <= 7) aoff[4] = off(kl0 + 1);
    }
    const Tc2Saved SV{B};
    float db1 = 0.f, db2 = 0.f, db3 = 0.f;
    uint32_t phase = 0;
    bool first = true;

    // cp.async of everything the forward saved for board bn into buffer `buf` (byte for byte; 16 bytes per copy)
    auto prefetch_board = [&](int64_t bn, int buf) {
        const uint32_t dst = in_addr + (uint32_t)buf * (uint32_t)sizeof(BoardIn);
        auto cp16 = [&](uint32_t d, const unsigned char *g) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(g) : "memory");
        };
        const unsigned char *g2 = SV.xt(saved, 1, bn), *g1 = SV.xt(saved, 0, bn), *ga = SV.a1t(saved, bn);
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            cp16(dst + (uint32_t)offsetof(BoardIn, xt2) + (uint32_t)(gtid + kBwdThreads * j) * 16u, g2 + (gtid + kBwdThreads * j) * 16);
            cp16(dst + (uint32_t)offsetof(BoardIn, xt1) + (uint32_t)(gtid + kBwdThreads * j) * 16u, g1 + (gtid + kBwdThreads * j) * 16);
        }
        // a1t (3072 B) and the coefficients (2592 B) are contiguous in the saved layout: 354 chunks of 16 B
        for (int c = gtid; c < (3072 + kV * 32) / 16; c += kBwdThreads)
            cp16(dst + (uint32_t)offsetof(BoardIn, a1t) + (uint32_t)c * 16u, ga + c * 16);
        asm volatile("cp.async.commit_group;\n" ::: "memory");
    };
    // ReLU mask of a layer from its saved activations: this thread's 48 nodes of its feature row of the tile -> 48 bits
    auto mask_from_tile = [&](const unsigned char *tile) -> u64 {
        u64 m = 0ull;
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            const int c8 = 6 * half + j;
            const uint4 ch = *reinterpret_cast<const uint4 *>(tile + row_off + (uint32_t)(c8 >> 2) * kFmBlock + (uint32_t)(((c8 & 3) ^ swz) << 4));
            m |= (u64)positive_bits_b(ch) << (8 * j);
        }
        return m;
    };
    // this thread's 48 values -> bf16 -> chunks 6 half .. 6 half + 5 of its row of sm.fm (nodes >= 81 written as zero: K padding of the dW MMAs)
    auto store_half_bf16 = [&](const float *z) {
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            const int c8 = 6 * half + j;
            uint4 v;
            if (c8 == 11) v = make_uint4(0u, 0u, 0u, 0u);                                  // nodes 88..95
            else if (c8 == 10) v = make_uint4(pack_bf16(z[8 * j], 0.f), 0u, 0u, 0u);       // node 80, then padding
            else v = pack8_bf16(z + 8 * j);
            *reinterpret_cast<uint4 *>(sm.fm + row_off + (uint32_t)(c8 >> 2) * kFmBlock + (uint32_t)(((c8 & 3) ^ swz) << 4)) = v;
        }
    };
    auto sync_then_issue_begin = [&]() {
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
        __syncthreads();
    };
    // The weight-gradient MMAs (dW3, dW2, dW1ext) produce nothing a thread reads before the end of the kernel: they are committed to
    // their own mbarrier and only waited for right before one of their operand buffers (the dZ tile, the saved-input buffer) is
    // overwritten, so they overlap the next phase.
    const uint32_t bar_w = smem_u32(&sm.mbar_w);
    uint32_t phase_w = 0;
    bool w_pending = false;
    auto wait_dw = [&]() {
        if (w_pending) {
            mbar_spin_b(bar_w, phase_w);
            phase_w ^= 1u;
            w_pending = false;
        }
    };
    auto wait_mma = [&]() {
        mbar_spin_b(bar, phase);
        phase ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    };

    int buf = 0;
    // launched programmatically: everything above (W^T tiles, zeroed adjacency, barriers, tensor-memory allocation) read only the parameters
    // and overlapped the tail of the heads backward; the saved activations and dg are read from here on
    aq_pdl_wait();
    prefetch_board(blockIdx.x, 0);
    uint4 mk_next = __ldcg(reinterpret_cast<const uint4 *>(SV.mask3(saved, blockIdx.x) + tid * 16));  // coherent: PDL rule (aq_common.cuh)
    float dg_next = __ldcg(dg + (int64_t)blockIdx.x * kH + tid);
#if TC2B_TIMING
    long long t_last = clock64();
#endif
    for (int64_t b = blockIdx.x; b < B; b += gridDim.x, buf ^= 1) {
        // ---- per-board inputs: wait for this board's saved tiles, start the next board's; masks, coefficients -> adjacency tile -------
        u64 m3, m2, m1;  // ReLU masks of this thread's 48 nodes
        // mask3 and dg of this board were requested one board ahead (two dependent-free global loads whose latency, ~900 cycles, sat
        // at the top of every board); the next board's are requested here
        const uint4 mk = mk_next;
        const float dgn = dg_next / (float)kV;  // d mean / d x_v
        if (b + gridDim.x < B) {
            mk_next = __ldcg(reinterpret_cast<const uint4 *>(SV.mask3(saved, b + gridDim.x) + tid * 16));
            dg_next = __ldcg(dg + (b + gridDim.x) * kH + tid);
        }
        m3 = half ? ((u64)(mk.y >> 16) | ((u64)mk.z << 16)) : ((u64)mk.x | ((u64)(mk.y & 0xFFFFu) << 32));
        TC2B_T(0);
        wait_dw();         // dW1ext of the previous board has read its A1^T tile (the buffer the prefetch below overwrites)
        asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        __syncthreads();   // the copies of every thread have landed; every thread is done with the other buffer (previous board)
        if (b + gridDim.x < B) prefetch_board(b + gridDim.x, buf ^ 1);
        const BoardIn &in = sm.in[buf];
        const uint32_t xt2_addr = in_addr + (uint32_t)buf * (uint32_t)sizeof(BoardIn), xt1_addr = xt2_addr + (uint32_t)offsetof(BoardIn, xt1);
        const uint32_t a1t_addr = xt2_addr + (uint32_t)offsetof(BoardIn, a1t);
        if (gtid < kV) {
            const float4 c0 = *reinterpret_cast<const float4 *>(in.coef + gtid * 8), c1 = *reinterpret_cast<const float4 *>(in.coef + gtid * 8 + 4);
            const float cv[5] = {c0.x, c0.y, c0.z, c0.w, c1.x};
#pragma unroll
            for (int k = 0; k < 5; ++k)
                if (aoff[k] != 0xFFFFFFFFu) *reinterpret_cast<float *>(sm.adj + aoff[k]) = cv[k];
        }
        TC2B_T(1);
        m2 = mask_from_tile(in.xt2);
        m1 = mask_from_tile(in.xt1);
        TC2B_T(2);
#pragma unroll 1
        for (int layer = 2; layer >= 1; --layer) {
            // ---- dY of layer (layer + 1): masked dX, written (back) into this thread's lane of the dX accumulator ----------------
            {
                float bsum = 0.f;
                uint32_t r[48];
                if (layer == 2) {
#pragma unroll
                    for (int i = 0; i < 48; ++i) r[i] = (m3 >> i) & 1ull ? __float_as_uint(dgn) : 0u;
                    bsum = (float)__popcll(m3) * dgn;
                } else {
                    float y[48];
                    tmem_ld48_b(lane_base + kColX + col0, y);
#pragma unroll
                    for (int i = 0; i < 48; ++i) {
                        const float t = (m2 >> i) & 1ull ? y[i] : 0.f;
                        bsum += t;
                        r[i] = __float_as_uint(t);
                    }
                }
                tmem_st48_b(lane_base + kColX + col0, r);
                asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
                if (layer == 2) db3 += bsum; else db2 += bsum;
            }
            TC2B_T(3);
            // ---- dZ^T = dY^T A_hat^T : tf32, A = the accumulator columns just written -------------------------------------------
            sync_then_issue_begin();
            if (issuer_warp) {
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                if (elect_one_lane()) {
#pragma unroll
                    for (int blk = 0; blk < 2; ++blk)
#pragma unroll
                        for (int s = 0; s < 8; ++s)  // 64 in-nodes = 8 K steps of 8 tf32
                            mma_ts_tf32_b(tmem + kColZ + blk * 48, tmem + kColX + blk * 32 + s * 8,
                                          desc_sw128(adj_addr + (uint32_t)blk * kAdjBlock + (uint32_t)(s >> 2) * kAdjKBlock + (uint32_t)(s & 3) * 32u),
                                          kIdescAgg, s ? 1u : 0u);
                    mma_commit(bar);
                }
                __syncwarp();
            }
            wait_mma();
            TC2B_T(4);
            // ---- dZ^T -> bf16 -> feature-major tile ----------------------------------------------------------------------------
            wait_dw();  // the previous weight-gradient MMA has read the tile
            {
                float z[48];
                tmem_ld48_b(lane_base + kColZ + col0, z);
                store_half_bf16(z);
            }
            TC2B_T(5);
            // ---- dX_{l}^T = W^T dZ^T (into the dX accumulator) and dW += dZ^T X ------------------------------------------------
            sync_then_issue_begin();
            if (issuer_warp) {
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                if (elect_one_lane()) {
                    const uint32_t wt = layer == 2 ? w3t_addr : w2t_addr;
#pragma unroll
                    for (int k = 0; k < 8; ++k)  // M = 128 (k_in), N = 96 (nodes), K = 128 (n_out): two 8-feature atoms of the tile per step
                        mma_bf16(tmem + kColX, desc_sw128(wt + (uint32_t)(k >> 2) * kRowBlock + (uint32_t)(k & 3) * 32u),
                                 desc_fm_mn_b(fm_addr + k * 1024), kIdescDX, k > 0 ? 1u : 0u);
                    mma_commit(bar);
                    const uint32_t accw = tmem + (layer == 2 ? kColW3 : kColW2);
#pragma unroll
                    for (int s = 0; s < 6; ++s)  // M = 128 (n_out), N = 128 (k_in), K = 96 (nodes): 32 B per step inside a 64 B node block
                        mma_bf16(accw, desc_fm_k_b(fm_addr + (uint32_t)(s >> 1) * kFmBlock + (uint32_t)(s & 1) * 32u),
                                 desc_fm_k_b((layer == 2 ? xt2_addr : xt1_addr) + (uint32_t)(s >> 1) * kFmBlock + (uint32_t)(s & 1) * 32u), kIdescDW, (first && s == 0) ? 0u : 1u);
                    mma_commit(bar_w);
                }
                __syncwarp();
            }
            w_pending = true;
            wait_mma();
            TC2B_T(6);
        }
        // ---- layer 1: dY1 = mask1 * dX1 -> bf16 tile;  dW1ext += dY1^T A1 ------------------------------------------------------------
        wait_dw();  // dW2 has read the tile
        {
            float bsum = 0.f;
            float y[48];
            tmem_ld48_b(lane_base + kColX + col0, y);
#pragma unroll
            for (int i = 0; i < 48; ++i) {
                y[i] = (m1 >> i) & 1ull ? y[i] : 0.f;
                bsum += y[i];
            }
            store_half_bf16(y);
            db1 += bsum;
        }
        TC2B_T(7);
        sync_then_issue_begin();
        if (issuer_warp) {
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            if (elect_one_lane()) {
#pragma unroll
                for (int s = 0; s < 6; ++s)  // M = 128, N = 16, K = 96
                    mma_bf16(tmem + kColW1, desc_fm_k_b(fm_addr + (uint32_t)(s >> 1) * kFmBlock + (uint32_t)(s & 1) * 32u),
                             desc_fm_k_b(a1t_addr + (uint32_t)(s >> 1) * 1024u + (uint32_t)(s & 1) * 32u), kIdescDW1, (first && s == 0) ? 0u : 1u);
                mma_commit(bar_w);
            }
            __syncwarp();
        }
        w_pending = true;
        TC2B_T(8);
        first = false;
        // (no barrier here: the next board starts with one, after its cp.async wait)
    }
    // ---- this CTA's partial gradients: accumulator rows -> its slot ---------------------------------------------
    wait_dw();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    {
        // dW2 (threads of half 0) / dW3 (half 1) rows leave through a per-warp transposing stage (the saved-input buffers are free now) so
        // that every global store is 32 consecutive floats of one row; a thread storing its own 32 columns touched 32 sectors per instruction
        float v[32];
        float *stage = reinterpret_cast<float *>(&sm.in[0]) + (gtid >> 5) * (32 * 33);
        float *bred = reinterpret_cast<float *>(sm.fm);  // [3][2][128]: the two halves' bias sums
        const int lane = gtid & 31, wrow = (tid >> 5) * 32;
        __syncthreads();  // every thread is past its last read of the tile and of the saved inputs
        bred[(0 * 2 + half) * 128 + tid] = db1;
        bred[(1 * 2 + half) * 128 + tid] = db2;
        bred[(2 * 2 + half) * 128 + tid] = db3;
#pragma unroll 1
        for (int cb = 0; cb < 4; ++cb) {
            tmem_ld32(lane_base + (half ? kColW3 : kColW2) + cb * 32, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) stage[lane * 33 + i] = v[i];
            __syncwarp();
            float *dst = slot + (half ? kOffW3 : kOffW2) + wrow * kH + cb * 32 + lane;
#pragma unroll 8
            for (int r = 0; r < 32; ++r) dst[r * kH] = stage[r * 33 + lane];
            __syncwarp();
        }
        __syncthreads();
        if (half == 0) {
            tmem_ld32(lane_base + kColW1, v);  // 16 columns used: [hi part (6) | lo part (6) | bias_hi | bias_lo | 0 | 0]
#pragma unroll
            for (int f = 0; f < kF; ++f) slot[kOffW1 + tid * kF + f] = v[f] + v[kF + f];  // both halves multiply W1
            slot[kOffB1 + tid] = bred[0 * 128 + tid] + bred[1 * 128 + tid];
            slot[kOffB2 + tid] = bred[2 * 128 + tid] + bred[3 * 128 + tid];
            slot[kOffB3 + tid] = bred[4 * 128 + tid] + bred[5 * 128 + tid];
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (gtid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(kTmemCols) : "memory");
}

}  // namespace

// partial: [kSlots = 148][64082] floats; this kernel fills the GCN ranges (W1,B1,W2,B2,W3,B3) of every slot
int aq_gcn_backward_tc2(const float *params, float *saved, const float *dg, int64_t B, float *partial, cudaStream_t st) {
    return aq_launch("gcn_backward_tc2_kernel", gcn_backward_tc2_kernel, dim3(148), kBwdThreads, sizeof(Bwd2Smem) + 1024, st, true, params, saved,
                     dg, B, partial);
}
