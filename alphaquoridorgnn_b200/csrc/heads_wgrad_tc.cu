// Weight gradients of the policy / value heads on the tensor cores (training, precision 1): dW = A^T B over the boards of the batch
// (reference train_network.py:87-89, loss.backward() through pv_network_gnn.py:38-51).
//   D0 [128 x 128] = [dhp | dhv]^T pooled      rows 0..63 = dWp0, rows 64..127 = dWv0        (+ column 128: the bias gradients)
//   D1 [256 x  64] = dz^T hp                   rows 0..208 = dWp2 (two M = 128 halves)          (+ column 64: dbp2)
//   dWv2 [64], dbv2 = du^T hv, sum(du)         on the CUDA cores (one output row)
// K = boards.  Both operands of a product are stored as the producer has them -- one row per board, the M (or N) index contiguous --
// i.e. MN-major for tcgen05.mma: bf16 tiles [32-wide MN blocks][K atoms of 8 boards][8][64 B], SWIZZLE_64B, the layout the trunk uses
// for its feature-major activations.  A "ones" column appended to each B operand makes the bias gradient (column sums of A over the
// boards) one more accumulator column.  One CTA per 64-board tile (kWgTile; grid-stride beyond 148 tiles), accumulators in tensor memory
// across the CTA's tiles, written once into the CTA's partial-gradient slot; the slot reduction that follows is the existing one.
// Replaces atb_jobs_kernel (FFMA, 39 us at B = 4,096) for the tensor-core training path; the fp32 path keeps atb_jobs_kernel.
#include <cstddef>
#include <cuda_bf16.h>
#include "aq_common.cuh"
#include "gnn_layout.cuh"
#include "tc_common.cuh"

using namespace aq;
using namespace aqtc;

namespace {

constexpr int kWgThreads = 512;
constexpr int kWgTile = 64;                         // boards per tile = K of one accumulation round (4 MMA steps of 16)
constexpr uint32_t kBlk = (kWgTile / 8) * 512;      // one 32-wide MN block: 8 K-atoms of [8 boards][64 B] = 4 KB
constexpr int kA0Blocks = 4, kB0Blocks = 5;         // [dhp | dhv] 128 wide; pooled 128 wide + the ones block
constexpr int kA1Blocks = 8, kB1Blocks = 3;         // dz 209 -> 256 wide; hp 64 wide + the ones block
constexpr uint32_t kN0 = 160, kN1 = 96;             // accumulator widths (multiples of 32: whole MN blocks of B)
constexpr uint32_t kColD0 = 0, kColD1a = kN0, kColD1b = kN0 + kN1;
constexpr uint32_t kWgTmemCols = 512;

struct WgSmem {
    unsigned char a0[kA0Blocks * kBlk];
    unsigned char b0[kB0Blocks * kBlk];
    unsigned char a1[kA1Blocks * kBlk];
    unsigned char b1[kB1Blocks * kBlk];
    float du[kWgTile];
    unsigned long long mbar;
    uint32_t tmem_base;
};
static_assert(sizeof(WgSmem) + 1024 <= 227 * 1024, "WgSmem exceeds shared memory");

// MN-major SWIZZLE_64B: LBO = stride between 32-wide MN blocks, SBO = stride between K atoms (8 boards)
__device__ __forceinline__ uint64_t desc_mn(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(kBlk >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
// byte offset of the 16-byte chunk holding MN elements [8 c, 8 c + 8) of board row r inside an operand tile
__device__ __forceinline__ uint32_t chunk_off(int r, int c) {
    return (uint32_t)(c >> 2) * kBlk + (uint32_t)(r >> 3) * 512u + (uint32_t)(r & 7) * 64u + (uint32_t)(((c & 3) ^ ((r & 7) >> 1)) << 4);
}
__device__ __forceinline__ uint4 pack8_bf16(const float *f) {
    uint4 v;
    v.x = pack_bf16(f[0], f[1]); v.y = pack_bf16(f[2], f[3]); v.z = pack_bf16(f[4], f[5]); v.w = pack_bf16(f[6], f[7]);
    return v;
}
__device__ __forceinline__ void tmem_ld16_wg(uint32_t taddr, float *v) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Rows [b0, b0 + 64) of a row-major fp32 matrix with 8 * kChunks columns -> bf16 operand tile, in two steps so that the loads of ALL
// operands of a tile are in flight before the first one is used (a load phase per operand costs a memory latency each).
// Coherent loads: the producers ran right before this kernel.
template <int kChunks>
struct TileRegs { float4 lo[kWgTile * kChunks / kWgThreads], hi[kWgTile * kChunks / kWgThreads]; };
template <int kChunks>
__device__ __forceinline__ void load_tile(TileRegs<kChunks> &t, const float *src, int64_t b0, int64_t B, int tid) {
    static_assert(kWgTile * kChunks % kWgThreads == 0, "chunks must divide evenly");
#pragma unroll
    for (int j = 0; j < kWgTile * kChunks / kWgThreads; ++j) {
        const int i = tid + j * kWgThreads, r = i / kChunks, c = i % kChunks;
        t.lo[j] = t.hi[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (b0 + r < B) {
            const float4 *p = reinterpret_cast<const float4 *>(src + (b0 + r) * (8 * kChunks) + c * 8);
            t.lo[j] = __ldcg(p);
            t.hi[j] = __ldcg(p + 1);
        }
    }
}
template <int kChunks>
__device__ __forceinline__ void store_tile(const TileRegs<kChunks> &t, unsigned char *tile, int col0_chunk, int tid) {
#pragma unroll
    for (int j = 0; j < kWgTile * kChunks / kWgThreads; ++j) {
        const int i = tid + j * kWgThreads, r = i / kChunks, c = i % kChunks;
        const float f[8] = {t.lo[j].x, t.lo[j].y, t.lo[j].z, t.lo[j].w, t.hi[j].x, t.hi[j].y, t.hi[j].z, t.hi[j].w};
        *reinterpret_cast<uint4 *>(tile + chunk_off(r, col0_chunk + c)) = pack8_bf16(f);
    }
}
// dz rows are 209 floats (not a multiple of 4): the 64 rows of a tile are read as one flat 16-byte-aligned range (64 x 209 floats =
// 3,344 float4) and every element is stored on its own (bf16, 2 bytes) at its (row, column) position.  Rows beyond B read as zero.
constexpr int kDzVec = kWgTile * kP / 4, kDzPer = (kDzVec + kWgThreads - 1) / kWgThreads;
__device__ __forceinline__ void load_dz(float4 *v, const float *dz, int64_t b0, int64_t B, int tid) {
    const int64_t limit = (B - b0 < kWgTile ? B - b0 : kWgTile) * kP;   // valid flat elements of this tile
    const float4 *src = reinterpret_cast<const float4 *>(dz + b0 * kP);
#pragma unroll
    for (int j = 0; j < kDzPer; ++j) {
        const int i = tid + j * kWgThreads;
        v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < kDzVec && (int64_t)i * 4 + 3 < limit) v[j] = __ldcg(src + i);
        else if (i < kDzVec) {   // the range ends inside this vector (last rows of the batch)
            const float *s = dz + b0 * kP + (int64_t)i * 4;
            if ((int64_t)i * 4 + 0 < limit) v[j].x = __ldcg(s);
            if ((int64_t)i * 4 + 1 < limit) v[j].y = __ldcg(s + 1);
            if ((int64_t)i * 4 + 2 < limit) v[j].z = __ldcg(s + 2);
        }
    }
}
__device__ __forceinline__ void store_dz(const float4 *v, unsigned char *tile, int tid) {
#pragma unroll
    for (int j = 0; j < kDzPer; ++j) {
        const int i = tid + j * kWgThreads;
        if (i >= kDzVec) continue;
        const float e[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
        int r = (i * 4) / kP, m = i * 4 - r * kP;   // row / column of the first element; the others follow, wrapping into the next row
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            *reinterpret_cast<__nv_bfloat16 *>(tile + chunk_off(r, m >> 3) + (m & 7) * 2) = __float2bfloat16_rn(e[k]);
            if (++m == kP) { m = 0; ++r; }
        }
    }
}

__global__ void __launch_bounds__(kWgThreads, 1)
heads_wgrad_tc_kernel(const float *dhp, const float *dhv, const float *dz, const float *du, const float *pooled, const float *hp,
                      const float *hv, int64_t B, float *__restrict__ partial) {
    extern __shared__ unsigned char smem_raw[];
    WgSmem &sm = *reinterpret_cast<WgSmem *>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int tid = threadIdx.x, warp = tid >> 5;
    aq_pdl_trigger();
    // ---- prologue (reads nothing the predecessors wrote): zero padding of the operand tiles, barrier, tensor memory ----------------
    {
        uint4 *z0 = reinterpret_cast<uint4 *>(sm.b0 + 4 * kBlk), *z1 = reinterpret_cast<uint4 *>(sm.b1 + 2 * kBlk);   // the ones blocks
        for (int i = tid; i < (int)(kBlk / 16); i += kWgThreads) { z0[i] = make_uint4(0u, 0u, 0u, 0u); z1[i] = make_uint4(0u, 0u, 0u, 0u); }
        uint4 *z2 = reinterpret_cast<uint4 *>(sm.a1 + 6 * kBlk);   // dz columns 192..255: only 192..208 are ever rewritten, the rest stays zero
        for (int i = tid; i < (int)(2 * kBlk / 16); i += kWgThreads) z2[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    const uint32_t bar = smem_u32(&sm.mbar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&sm.tmem_base)), "r"(kWgTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem = sm.tmem_base;
    aq_pdl_wait();   // dhp, dhv, dz, du (heads backward) and the saved activations are complete from here on

    // instruction descriptors: D = f32, A = B = bf16, both operands MN-major (bits 15, 16), M = 128
    constexpr uint32_t kIdesc0 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((kN0 >> 3) << 17) | ((128u >> 4) << 24);
    constexpr uint32_t kIdesc1 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((kN1 >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t a0 = smem_u32(sm.a0), b0a = smem_u32(sm.b0), a1 = smem_u32(sm.a1), b1a = smem_u32(sm.b1);
    const int64_t ntiles = (B + kWgTile - 1) / kWgTile;
    uint32_t phase = 0;
    float wv2 = 0.f, sdu = 0.f;   // this thread's part of dWv2[tid % 64] and of dbv2
    bool first = true;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t r0 = t * kWgTile;
        if (!first) {   // the previous tile's MMAs have read the operand tiles, its value-row loop the du values
            __syncthreads();
            uint32_t ok = 0;
            while (!ok)
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                             : "=r"(ok) : "r"(bar), "r"(phase) : "memory");
            phase ^= 1u;
        }
        {
            float4 vz[kDzPer];
            TileRegs<kH / 8> tp;
            TileRegs<kHH / 8> t0, t1, t2;
            load_dz(vz, dz, r0, B, tid);
            load_tile(tp, pooled, r0, B, tid);
            load_tile(t0, dhp, r0, B, tid);
            load_tile(t1, dhv, r0, B, tid);
            load_tile(t2, hp, r0, B, tid);
            store_dz(vz, sm.a1, tid);
            store_tile(tp, sm.b0, 0, tid);
            store_tile(t0, sm.a0, 0, tid);
            store_tile(t1, sm.a0, kHH / 8, tid);
            store_tile(t2, sm.b1, 0, tid);
        }
        if (tid < kWgTile) {   // the ones column: 1 for the boards that exist (bias gradient = sum over boards), and du for the value row
            const bool on = r0 + tid < B;
            const uint4 one = make_uint4(on ? 0x00003F80u : 0u, 0u, 0u, 0u);   // bf16 {1, 0, 0, 0, 0, 0, 0, 0}
            *reinterpret_cast<uint4 *>(sm.b0 + chunk_off(tid, 16)) = one;
            *reinterpret_cast<uint4 *>(sm.b1 + chunk_off(tid, 8)) = one;
            sm.du[tid] = on ? __ldcg(du + r0 + tid) : 0.f;
        }
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
        __syncthreads();
        if (warp == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            if (elect_one_lane()) {
#pragma unroll
                for (uint32_t k = 0; k < kWgTile / 16; ++k) {   // 16 boards = two K atoms = 1,024 B inside every MN block
                    const uint32_t acc = (!first || k > 0) ? 1u : 0u;
                    mma_bf16(tmem + kColD0, desc_mn(a0 + k * 1024u), desc_mn(b0a + k * 1024u), kIdesc0, acc);
                    mma_bf16(tmem + kColD1a, desc_mn(a1 + k * 1024u), desc_mn(b1a + k * 1024u), kIdesc1, acc);
                    mma_bf16(tmem + kColD1b, desc_mn(a1 + 4u * kBlk + k * 1024u), desc_mn(b1a + k * 1024u), kIdesc1, acc);
                }
                mma_commit(bar);
            }
            __syncwarp();
        }
        // value head's output layer (one row), while the MMAs run: dWv2[n] += sum_r du[r] hv[r][n], dbv2 += sum_r du[r].  Thread
        // (n = tid % 64, part = tid / 64) takes 8 boards: its 8 loads are all in flight at once; the parts meet at the end.
        {
            constexpr int kRows = kWgTile / (kWgThreads / kHH);
            const int n = tid & (kHH - 1), part = tid >> 6;
            float h[kRows];
#pragma unroll
            for (int i = 0; i < kRows; ++i) {
                const int64_t b = r0 + part * kRows + i;
                h[i] = b < B ? __ldcg(hv + b * kHH + n) : 0.f;
            }
#pragma unroll
            for (int i = 0; i < kRows; ++i) {
                const float d = sm.du[part * kRows + i];   // zero beyond B
                wv2 = fmaf(d, h[i], wv2);
                sdu += d;
            }
        }
        first = false;
    }
    // ---- accumulators -> this CTA's partial slot ---------------------------------------------------------------------------------
    {
        uint32_t ok = 0;
        while (!ok)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                         : "=r"(ok) : "r"(bar), "r"(phase) : "memory");
    }
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    float *slot = partial + (int64_t)blockIdx.x * kNumParams;
    const int m = tid & 127, q = tid >> 7;                                   // accumulator row (TMEM lane) / column quarter
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);   // this warp's TMEM lane quadrant
    // Every store instruction writes consecutive floats of one output row: the warp's 32 lanes x 32 (16) columns go through a
    // per-warp transposing stage in shared memory (the operand tiles are free: every MMA has completed).  Writing the accumulator
    // rows straight from the lanes touches 32 sectors per instruction and made this epilogue two thirds of the kernel.
    static_assert(kWgThreads / 32 * 32 * 33 * 4 <= sizeof(WgSmem::a0) + sizeof(WgSmem::b0) + sizeof(WgSmem::a1) + sizeof(WgSmem::b1), "staging area");
    float *stage = reinterpret_cast<float *>(sm.a0) + warp * (32 * 33);   // a0 | b0 | a1 | b1 are contiguous
    const int lane = tid & 31, mq = (warp & 3) * 32;   // first accumulator row of this warp's lane quadrant
    {   // D0: 128 columns, 32 per quarter; rows 0..63 -> dWp0, 64..127 -> dWv0
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float v[16];
            tmem_ld16_wg(lane_base + kColD0 + q * 32 + h * 16, v);
#pragma unroll
            for (int i = 0; i < 16; ++i) stage[lane * 33 + h * 16 + i] = v[i];
        }
        __syncwarp();
#pragma unroll 4
        for (int r = 0; r < 32; ++r) {
            const int row = mq + r;
            float *dst = slot + (row < kHH ? kOffWP0 + row * kH : kOffWV0 + (row - kHH) * kH) + q * 32;
            dst[lane] = stage[r * 33 + lane];
        }
        __syncwarp();
    }
#pragma unroll
    for (int half = 0; half < 2; ++half) {   // D1: 64 columns, 16 per quarter; rows 0..127 (a) and 128..208 (b) of dWp2
        float v[16];
        tmem_ld16_wg(lane_base + (half ? kColD1b : kColD1a) + q * 16, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) stage[lane * 17 + i] = v[i];
        __syncwarp();
#pragma unroll 4
        for (int r2 = 0; r2 < 16; ++r2) {   // two rows per instruction, 16 consecutive floats each
            const int r = 2 * r2 + (lane >> 4), row = half * 128 + mq + r;
            if (row < kP) slot[kOffWP2 + row * kHH + q * 16 + (lane & 15)] = stage[r * 17 + (lane & 15)];
        }
        __syncwarp();
    }
    {   // bias gradients: the ones columns (128 of D0, 64 of D1); quarter 0 writes dbp0 / dbv0, quarter 1 dbp2 rows 0..127, quarter 2 the rest
        float v[16];
        tmem_ld16_wg(lane_base + (q == 0 ? kColD0 + 128u : q == 1 ? kColD1a + 64u : kColD1b + 64u), v);
        if (q == 0) slot[m < kHH ? kOffBP0 + m : kOffBV0 + (m - kHH)] = v[0];
        else if (q == 1) slot[kOffBP2 + m] = v[0];
        else if (q == 2 && m + 128 < kP) slot[kOffBP2 + m + 128] = v[0];
    }
    {   // the eight parts of the value row meet in shared memory (the operand tiles are free: every MMA has completed)
        float *red = reinterpret_cast<float *>(sm.a0);
        __syncthreads();   // every warp is done with its staging area
        red[tid] = wv2;
        if ((tid & (kHH - 1)) == 0) red[kWgThreads + (tid >> 6)] = sdu;
        __syncthreads();
        if (tid < kHH) {
            float t = 0.f;
#pragma unroll
            for (int p = 0; p < kWgThreads / kHH; ++p) t += red[p * kHH + tid];
            slot[kOffWV2 + tid] = t;
        } else if (tid == kHH) {
            float t = 0.f;
#pragma unroll
            for (int p = 0; p < kWgThreads / kHH; ++p) t += red[kWgThreads + p];
            slot[kOffBV2] = t;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(kWgTmemCols) : "memory");
}

}  // namespace

// Number of partial slots the kernel fills (= its grid): one per 64-board tile (kWgTile), at most one per SM.
int aq_heads_wgrad_tc_slots(int64_t B) {
    const int64_t tiles = (B + kWgTile - 1) / kWgTile;
    return (int)(tiles < 148 ? tiles : 148);
}

int aq_heads_wgrad_tc(const float *dhp, const float *dhv, const float *dz, const float *du, const float *pooled, const float *hp,
                      const float *hv, int64_t B, float *partial, cudaStream_t st) {
    const int slots = aq_heads_wgrad_tc_slots(B);
    if (slots <= 0) return 0;
    return aq_launch("heads_wgrad_tc_kernel", heads_wgrad_tc_kernel, (unsigned)slots, kWgThreads, sizeof(WgSmem) + 1024, st, true, dhp, dhv, dz,
                     du, pooled, hp, hv, B, partial);
}
