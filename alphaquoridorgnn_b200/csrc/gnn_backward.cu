// Backward of GraphPolicyValueNetwork (autograd of train_network.py:93) -- fp32, atomic-free and
// deterministic.  A_hat is symmetric (is_wall_blocking is symmetric, game_logic.py:145-167), so the
// transposed-CSR scatter of the backward pass is the same 5-point gather as the forward.
//   heads_backward_kernel : softmax/tanh/MLP backward per board -> dz, dhp, dhv, du, dg
//   gcn_backward_kernel   : per board dY_l, dZ_l = A_hat dY_l, dX_{l-1} = dZ_l W_l ; bias partials
//   atb_jobs_kernel       : all weight gradients dW = A^T B as split-row partial GEMMs (one launch)
//   reduce_partials_kernel: grads[i] = sum over slots of partial[slot][i]
// plus the loss gradient of train_network.py:54-55,85-89 and the Adam step.
#include <algorithm>
#include <cstdlib>
#include "gnn_fp32.cuh"

using namespace aq;

constexpr int kSlots = 148;  // partial-gradient slots (one per persistent CTA / row chunk)

struct BwdWs {
    int64_t B;
    __host__ __device__ int64_t dz3() const { return 0; }
    __host__ __device__ int64_t dz2() const { return B * kV * kH; }
    __host__ __device__ int64_t dy1() const { return 2 * B * kV * kH; }
    __host__ __device__ int64_t dg() const { return 3 * B * kV * kH; }
    __host__ __device__ int64_t dhp() const { return dg() + B * kH; }
    __host__ __device__ int64_t dhv() const { return dhp() + B * kHH; }
    __host__ __device__ int64_t dz() const { return dhv() + B * kHH; }
    __host__ __device__ int64_t du() const { return dz() + B * kP; }
    __host__ __device__ int64_t partial() const { return (du() + B + 3) / 4 * 4; }
    __host__ __device__ int64_t total() const { return partial() + (int64_t)kSlots * kNumParams; }
};

// ------------------------------------------------------------------------------------------
// heads backward: one warp per board
// ------------------------------------------------------------------------------------------
constexpr int kHbThreads = 512;  // at most 16 warps = 16 boards in flight per CTA (launched with 8 warps for small batches, where the weight fill dominates)
// kNB boards per warp at a time: the three contractions of a board are bound by shared-memory reads of the weights (one LDS per
// FMA when a warp owns one board); with kNB boards every weight value read feeds kNB FMAs.  kNB is chosen by the batch size so that
// the warps of the machine still get one group each (1 up to 2,367 boards, 2 up to 8,191, 4 above).
template <int kNB>
struct HeadBwdSmem {
    float wp2[kP * kHH];  // [a][j]
    float wp0[kHH * kH];  // [j][k]
    float wv0[kHH * kH];
    float wv2[kHH];
    float dz[kHbThreads / 32][kNB][224];
    float dh[kHbThreads / 32][kNB][2 * kHH];  // dhp | dhv
};
static_assert(sizeof(HeadBwdSmem<4>) <= 227 * 1024, "HeadBwdSmem too large");

// kLoss: the loss gradient of train_network.py:54-55,85-89 (loss_grad_kernel below, same expressions in the same order) is computed
// here from the saved network outputs and the targets instead of being read from dpolicy / dvalue: one launch and one
// [B,209] round trip less per training step.
template <bool kLoss, int kNB>
__global__ void __launch_bounds__(kHbThreads, 1)
heads_backward_kernel(const float *__restrict__ params, const float *saved,   // saved: written by the kernel this one may overlap -- no __restrict__ (PDL rule)
                      const float *dpolicy, const float *dvalue, const float *__restrict__ ptarget, const float *__restrict__ vtarget,
                      float inv_total, float *__restrict__ loss, int64_t B, float *__restrict__ ws) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    HeadBwdSmem<kNB> &sm = *reinterpret_cast<HeadBwdSmem<kNB> *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    aq_pdl_trigger();  // the trunk backward may be scheduled as SMs free up; it waits for this grid before it reads dg
    // 116 KB of head weights per CTA: 16-byte loads where the parameter offset allows it, 8 loads in flight per thread
    static_assert(kOffWP2 % 4 == 0 && kOffWP0 % 4 == 0 && (kP * kHH) % 4 == 0, "float4 fill");
#pragma unroll 8
    for (int i = tid; i < kP * kHH / 4; i += (int)blockDim.x)
        reinterpret_cast<float4 *>(sm.wp2)[i] = __ldg(reinterpret_cast<const float4 *>(params + kOffWP2) + i);
#pragma unroll 8
    for (int i = tid; i < kHH * kH / 4; i += (int)blockDim.x)
        reinterpret_cast<float4 *>(sm.wp0)[i] = __ldg(reinterpret_cast<const float4 *>(params + kOffWP0) + i);
#pragma unroll 8
    for (int i = tid; i < kHH * kH; i += (int)blockDim.x) sm.wv0[i] = __ldg(params + kOffWV0 + i);
    if (tid < kHH) sm.wv2[tid] = __ldg(params + kOffWV2 + tid);
    aq_pdl_wait();     // launched programmatically: the weight fill above overlaps the tail of the loss kernel; dpolicy / dvalue are read below
    __syncthreads();
    const SavedLayout L{B};
    const BwdWs W{B};
    const int nwarps = (int)blockDim.x >> 5;
    float loss_p = 0.f, loss_v = 0.f;
    for (int64_t b0 = ((int64_t)blockIdx.x * nwarps + warp) * kNB; b0 < B; b0 += (int64_t)gridDim.x * nwarps * kNB) {
        __syncwarp();
        float du_[kNB];
        // ---- per board: loss gradient (or the given one), softmax backward dz = p * (dp - sum_j dp_j p_j) -> shared memory ----
#pragma unroll
        for (int nb = 0; nb < kNB; ++nb) {
            const int64_t b = b0 + nb;
            du_[nb] = 0.f;
            if (b >= B) {   // a group's tail: zero rows contribute nothing to the blocked contractions below
#pragma unroll
                for (int t = 0; t < 7; ++t) sm.dz[warp][nb][lane + 32 * t] = 0.f;
                continue;
            }
            float p[7], dp[7], s = 0.f;
            float dval;
            if (kLoss) {
                // CrossEntropyLoss(input = softmax probabilities, target = probabilities): -sum_a t_a log_softmax(p)_a -- the second
                // softmax is the reference's behaviour -- and MSELoss, both 'mean' over the global batch
                float tg[7], mx = -INFINITY;
#pragma unroll
                for (int t = 0; t < 7; ++t) {
                    const int a = lane + 32 * t;
                    p[t] = a < kP ? __ldcg(saved + L.policy() + b * kP + a) : -INFINITY;
                    tg[t] = a < kP ? __ldg(ptarget + b * kP + a) : 0.f;
                    mx = fmaxf(mx, p[t]);
                }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
                float se = 0.f, tsum = 0.f;
#pragma unroll
                for (int t = 0; t < 7; ++t) {
                    if (lane + 32 * t < kP) se += expf(p[t] - mx);
                    tsum += tg[t];
                }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) {
                    se += __shfl_xor_sync(0xffffffffu, se, d);
                    tsum += __shfl_xor_sync(0xffffffffu, tsum, d);
                }
                const float lse = mx + logf(se);
                float l = 0.f;
#pragma unroll
                for (int t = 0; t < 7; ++t) {
                    if (lane + 32 * t < kP) {
                        const float ls = p[t] - lse;
                        l -= tg[t] * ls;
                        dp[t] = (expf(ls) * tsum - tg[t]) * inv_total;
                    } else {
                        p[t] = 0.f;
                        dp[t] = 0.f;
                    }
                    s = fmaf(dp[t], p[t], s);
                }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) l += __shfl_xor_sync(0xffffffffu, l, d);
                const float dv0 = __ldcg(saved + L.value() + b) - __ldg(vtarget + b);
                dval = 2.f * dv0 * inv_total;
                loss_p += l;
                loss_v += dv0 * dv0;
            } else {
#pragma unroll
                for (int t = 0; t < 7; ++t) {
                    const int a = lane + 32 * t;
                    p[t] = a < kP ? saved[L.policy() + b * kP + a] : 0.f;
                    dp[t] = a < kP ? __ldcg(dpolicy + b * kP + a) : 0.f;  // written by the loss kernel this grid may overlap: coherent load (PDL rule, aq_common.cuh)
                    s = fmaf(dp[t], p[t], s);
                }
                dval = __ldcg(dvalue + b);
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
#pragma unroll
            for (int t = 0; t < 7; ++t) {
                const int a = lane + 32 * t;
                const float dz = p[t] * (dp[t] - s);
                sm.dz[warp][nb][a] = dz;
                if (a < kP) ws[W.dz() + b * kP + a] = dz;
            }
            // value head: v = tanh(u); du = dv * (1 - v^2)
            const float v = saved[L.value() + b];
            du_[nb] = dval * (1.f - v * v);
        }
        __syncwarp();
        // ---- dhp = (Wp2^T dz) * (hp > 0) for the kNB boards at once; outputs j = lane, lane+32 ----
        float h0[kNB], h1[kNB];
#pragma unroll
        for (int nb = 0; nb < kNB; ++nb) h0[nb] = h1[nb] = 0.f;
#pragma unroll 4
        for (int a = 0; a < kP; ++a) {
            const float w0 = sm.wp2[a * kHH + lane], w1 = sm.wp2[a * kHH + lane + 32];
#pragma unroll
            for (int nb = 0; nb < kNB; ++nb) {
                const float dz = sm.dz[warp][nb][a];
                h0[nb] = fmaf(dz, w0, h0[nb]);
                h1[nb] = fmaf(dz, w1, h1[nb]);
            }
        }
#pragma unroll
        for (int nb = 0; nb < kNB; ++nb) {
            const int64_t b = b0 + nb;
            float a0 = 0.f, a1 = 0.f, g0 = 0.f, g1 = 0.f;
            if (b < B) {
                const float hp0 = saved[L.hp() + b * kHH + lane], hp1 = saved[L.hp() + b * kHH + lane + 32];
                a0 = hp0 > 0.f ? h0[nb] : 0.f;
                a1 = hp1 > 0.f ? h1[nb] : 0.f;
                // dhv = du * wv2 * (hv > 0)
                const float hv0 = saved[L.hv() + b * kHH + lane], hv1 = saved[L.hv() + b * kHH + lane + 32];
                g0 = hv0 > 0.f ? du_[nb] * sm.wv2[lane] : 0.f;
                g1 = hv1 > 0.f ? du_[nb] * sm.wv2[lane + 32] : 0.f;
                ws[W.dhp() + b * kHH + lane] = a0; ws[W.dhp() + b * kHH + lane + 32] = a1;
                ws[W.dhv() + b * kHH + lane] = g0; ws[W.dhv() + b * kHH + lane + 32] = g1;
                if (lane == 0) ws[W.du() + b] = du_[nb];
            }
            sm.dh[warp][nb][lane] = a0; sm.dh[warp][nb][lane + 32] = a1;
            sm.dh[warp][nb][kHH + lane] = g0; sm.dh[warp][nb][kHH + lane + 32] = g1;
        }
        __syncwarp();
        // ---- dg = Wp0^T dhp + Wv0^T dhv for the kNB boards at once; outputs k = lane + 32 t ----
        float dg[kNB][4];
#pragma unroll
        for (int nb = 0; nb < kNB; ++nb)
#pragma unroll
            for (int t = 0; t < 4; ++t) dg[nb][t] = 0.f;
#pragma unroll 2
        for (int j = 0; j < kHH; ++j) {
            float wa[4], wc[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) { wa[t] = sm.wp0[j * kH + lane + 32 * t]; wc[t] = sm.wv0[j * kH + lane + 32 * t]; }
#pragma unroll
            for (int nb = 0; nb < kNB; ++nb) {
                const float a = sm.dh[warp][nb][j], c = sm.dh[warp][nb][kHH + j];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    dg[nb][t] = fmaf(a, wa[t], dg[nb][t]);
                    dg[nb][t] = fmaf(c, wc[t], dg[nb][t]);
                }
            }
        }
#pragma unroll
        for (int nb = 0; nb < kNB; ++nb)
            if (b0 + nb < B) {
#pragma unroll
                for (int t = 0; t < 4; ++t) ws[W.dg() + (b0 + nb) * kH + lane + 32 * t] = dg[nb][t];
            }
    }
    if (kLoss && loss) {  // monitoring scalars: one pair of atomics per CTA
        __shared__ float red[2][kHbThreads / 32];
        if (lane == 0) { red[0][warp] = loss_p; red[1][warp] = loss_v; }
        __syncthreads();
        if (warp == 0) {
            float a = lane < nwarps ? red[0][lane] : 0.f, c = lane < nwarps ? red[1][lane] : 0.f;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                a += __shfl_xor_sync(0xffffffffu, a, d);
                c += __shfl_xor_sync(0xffffffffu, c, d);
            }
            if (lane == 0) {
                atomicAdd(loss + 0, a * inv_total);
                atomicAdd(loss + 1, c * inv_total);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// GCN backward: one board per CTA iteration
// ------------------------------------------------------------------------------------------
struct GcnBwdSmem {
    float w2[kH * kH];  // natural [n][k]: dX = dZ W reduces over n
    float w3[kH * kH];
    float bufa[kV * kH];
    float bufb[kV * kH];
    float pad[7 * kH];  // GEMM over-read of bufb rows 81..87
    float coef[kV * 5 + 3];
    float dg[kH];
    float red[256];
};
static_assert(sizeof(GcnBwdSmem) <= 227 * 1024, "GcnBwdSmem too large");

__device__ __forceinline__ void colsum_accumulate(const float *buf, float &acc, int tid) {
    const int n = tid & (kH - 1);
    float s = 0.f;
    for (int v = tid >> 7; v < kV; v += 2) s += buf[v * kH + n];
    acc += s;
}

__global__ void __launch_bounds__(kGcnThreads, 1)
gcn_backward_kernel(const float *__restrict__ params, const float *__restrict__ saved, int64_t B,
                    float *__restrict__ ws) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    GcnBwdSmem &sm = *reinterpret_cast<GcnBwdSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const SavedLayout L{B};
    const BwdWs W{B};
    float db1 = 0.f, db2 = 0.f, db3 = 0.f;  // per-thread partial column sums (column tid & 127)
    if ((int64_t)blockIdx.x < B) {
        load_weight_natural(sm.w2, params + kOffW2, tid);
        load_weight_natural(sm.w3, params + kOffW3, tid);
    }
    for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
        __syncthreads();
        for (int i = tid; i < kV * 5; i += kGcnThreads) sm.coef[i] = saved[L.coef() + b * kV * 5 + i];
        if (tid < kH) sm.dg[tid] = ws[W.dg() + b * kH + tid] / (float)kV;  // d mean / d x_v
        __syncthreads();
        // dY3 = (X3 > 0) * dg/81
        {
            const float4 *x3 = reinterpret_cast<const float4 *>(saved + L.x(2) + b * kV * kH);
            const float4 d = reinterpret_cast<const float4 *>(sm.dg)[lane];
            for (int i = tid; i < kV * kH / 4; i += kGcnThreads) {  // i & 31 == lane
                const float4 x = x3[i];
                reinterpret_cast<float4 *>(sm.bufa)[i] = make_float4(x.x > 0.f ? d.x : 0.f, x.y > 0.f ? d.y : 0.f,
                                                                     x.z > 0.f ? d.z : 0.f, x.w > 0.f ? d.w : 0.f);
            }
        }
        __syncthreads();
#pragma unroll 1
        for (int layer = 2; layer >= 1; --layer) {
            // bufa = dY_{layer+1}; bias gradient and dZ = A_hat dY
            colsum_accumulate(sm.bufa, layer == 2 ? db3 : db2, tid);
            aggregate<false>(sm.bufa, sm.bufb, sm.coef, nullptr, warp, lane);
            __syncthreads();
            {
                float4 *dst = reinterpret_cast<float4 *>(ws + (layer == 2 ? W.dz3() : W.dz2()) + b * kV * kH);
                const float4 *src = reinterpret_cast<const float4 *>(sm.bufb);
                for (int i = tid; i < kV * kH / 4; i += kGcnThreads) dst[i] = src[i];
            }
            // dX_layer = dZ W ; dY_layer = (X_layer > 0) * dX_layer
            float acc[kRowsPerWarp][4];
            gemm_rows(sm.bufb, layer == 2 ? sm.w3 : sm.w2, warp, lane, acc);
            const float4 *xl = reinterpret_cast<const float4 *>(saved + L.x(layer - 1) + b * kV * kH);
#pragma unroll
            for (int i = 0; i < kRowsPerWarp; ++i) {
                const int r = warp * kRowsPerWarp + i;
                if (r < kV) {
                    const float4 x = xl[r * 32 + lane];
                    reinterpret_cast<float4 *>(sm.bufa)[r * 32 + lane] =
                        make_float4(x.x > 0.f ? acc[i][0] : 0.f, x.y > 0.f ? acc[i][1] : 0.f,
                                    x.z > 0.f ? acc[i][2] : 0.f, x.w > 0.f ? acc[i][3] : 0.f);
                }
            }
            __syncthreads();
        }
        // bufa = dY1: bias gradient, and keep it for dW1 = dY1^T (A_hat X0)
        colsum_accumulate(sm.bufa, db1, tid);
        {
            float4 *dst = reinterpret_cast<float4 *>(ws + W.dy1() + b * kV * kH);
            const float4 *src = reinterpret_cast<const float4 *>(sm.bufa);
            for (int i = tid; i < kV * kH / 4; i += kGcnThreads) dst[i] = src[i];
        }
    }
    // bias partials of this CTA (zeros when it had no board): combine the two row halves
    float *slot = ws + W.partial() + (int64_t)blockIdx.x * kNumParams;
    const int n = tid & (kH - 1);
    float vals[3] = {db1, db2, db3};
    const int offs[3] = {kOffB1, kOffB2, kOffB3};
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        __syncthreads();
        sm.red[tid] = vals[q];
        __syncthreads();
        if (tid < kH) slot[offs[q] + n] = sm.red[tid] + sm.red[tid + kH];
    }
}

// ------------------------------------------------------------------------------------------
// weight gradients: out[m][n] = sum_r A[r][m] * Bm[r][n], rows split over J.nslots chunks (slot s of the partial buffer).
// One launch for all jobs: grid = (max nslots, kMaxMTiles, njobs).  The node-level jobs of the fp32 path (R = 81 B rows)
// use all kSlots chunks; the head jobs (R = B rows) use one chunk per 64 boards -- every chunk writes a full [M][N] tile
// that reduce_partials_kernel reads back, so chunks that would hold a handful of rows are pure overhead.
// ------------------------------------------------------------------------------------------
struct AtbJob {
    const float *A; int lda; int M;
    const float *Bm; int ldb; int N;  // Bm == nullptr: implicit ones, N = 1 (column sums of A)
    int64_t R;
    int out_off;                      // offset inside a partial slot, row-major [M][N]
    int nslots;                       // row chunks = partial slots this job fills
    int bias_off;                     // >= 0: also write the column sums of A (the bias gradient of the same layer) there
};
constexpr int kMaxJobs = 12;
struct AtbJobs { AtbJob job[kMaxJobs]; int n; };
constexpr int kAtbMT = 64, kAtbKT = 32, kMaxMTiles = 4;

__global__ void __launch_bounds__(256)
atb_jobs_kernel(const AtbJobs jobs, float *__restrict__ partial) {
    aq_pdl_trigger();
    aq_pdl_wait();  // everything this kernel reads was written by the backward kernels before it
    const AtbJob J = jobs.job[blockIdx.z];
    const int m0 = blockIdx.y * kAtbMT;
    if (m0 >= J.M || (int)blockIdx.x >= J.nslots) return;
    __shared__ __align__(16) float As[kAtbKT][kAtbMT];
    __shared__ __align__(16) float Bs[kAtbKT][kH];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;  // tx -> 8 columns, ty -> 4 rows of the tile
    const int64_t per = (J.R + J.nslots - 1) / J.nslots;
    const int64_t r_begin = (int64_t)blockIdx.x * per;
    const int64_t r_end = r_begin + per < J.R ? r_begin + per : J.R;
    float acc[4][8];
    float bias_acc = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    for (int64_t r0 = r_begin; r0 < r_end; r0 += kAtbKT) {
        // all global loads of the tile are issued before the first use (24 independent loads per thread in flight; a load
        // per loop iteration with its own bounds test serialised their latencies: 50 us for 0.2 GFLOP)
        float av_[kAtbKT * kAtbMT / 256], bv_[kAtbKT * kH / 256];
#pragma unroll
        for (int j = 0; j < kAtbKT * kAtbMT / 256; ++j) {
            const int i = tid + 256 * j, k = i / kAtbMT, m = i % kAtbMT;
            const int64_t r = r0 + k;
            av_[j] = (r < r_end && m0 + m < J.M) ? __ldcg(J.A + r * J.lda + m0 + m) : 0.f;  // coherent loads: PDL rule (aq_common.cuh)
        }
#pragma unroll
        for (int j = 0; j < kAtbKT * kH / 256; ++j) {
            const int i = tid + 256 * j, k = i / kH, n = i % kH;
            const int64_t r = r0 + k;
            float v = 0.f;
            if (r < r_end && n < J.N) v = J.Bm ? __ldcg(J.Bm + r * J.ldb + n) : 1.f;
            bv_[j] = v;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kAtbKT * kAtbMT / 256; ++j) {
            const int i = tid + 256 * j;
            As[i / kAtbMT][i % kAtbMT] = av_[j];
        }
#pragma unroll
        for (int j = 0; j < kAtbKT * kH / 256; ++j) {
            const int i = tid + 256 * j;
            Bs[i / kH][i % kH] = bv_[j];
        }
        __syncthreads();
        if (J.bias_off >= 0 && tid < kAtbMT) {  // bias gradient = column sums of A: two warps, one column each
            float t = 0.f;
#pragma unroll
            for (int k = 0; k < kAtbKT; ++k) t += As[k][tid];
            bias_acc += t;
        }
#pragma unroll 8
        for (int k = 0; k < kAtbKT; ++k) {
            const float4 a = *reinterpret_cast<const float4 *>(&As[k][ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 8]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 8 + 4]);
            const float av[4] = {a.x, a.y, a.z, a.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
    }
    if (J.bias_off >= 0 && tid < kAtbMT && m0 + tid < J.M) partial[(int64_t)blockIdx.x * kNumParams + J.bias_off + m0 + tid] = bias_acc;
    float *slot = partial + (int64_t)blockIdx.x * kNumParams + J.out_off;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= J.M) continue;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = tx * 8 + j;
            if (n < J.N) slot[m * J.N + n] = acc[i][j];
        }
    }
}

// grads[i] = sum over the slots that hold parameter i (GCN ranges: kSlots; head ranges, i >= kOffWP0: head_slots).
// block = 128 parameter pairs x 4 slot groups: group g adds slots g, g+4, g+8, ... in that order and the four group sums are
// combined as (g0 + g1) + (g2 + g3) -- a fixed order, so the result is deterministic -- with 4 x 4 independent 8-byte loads
// in flight per thread (the slot stride, 64082 floats, is 8-byte but not 16-byte aligned).
constexpr int kRedPairs = 128;
__global__ void __launch_bounds__(kRedPairs * 4)
reduce_partials_kernel(const float *partial, float *__restrict__ grads, int head_slots) {
    __shared__ float2 part[4][kRedPairs];
    aq_pdl_wait();
    const int tx = threadIdx.x & (kRedPairs - 1), g = threadIdx.x / kRedPairs;
    const int i = 2 * (blockIdx.x * kRedPairs + tx);  // kNumParams is even
    float2 s = make_float2(0.f, 0.f);
    if (i < kNumParams) {
        // a pair never straddles the GCN / head boundary (kOffWP0 is even)
        const int n = i >= kOffWP0 ? head_slots : kSlots;
        const float *src = partial + i;
#pragma unroll 4
        for (int k = g; k < n; k += 4) {
            const float2 v = __ldcg(reinterpret_cast<const float2 *>(src + (int64_t)k * kNumParams));  // coherent: PDL rule
            s.x += v.x; s.y += v.y;
        }
    }
    part[g][tx] = s;
    __syncthreads();
    if (g == 0 && i < kNumParams) {
        const float2 a = part[0][tx], b = part[1][tx], c = part[2][tx], d = part[3][tx];
        *reinterpret_cast<float2 *>(grads + i) = make_float2((a.x + b.x) + (c.x + d.x), (a.y + b.y) + (c.y + d.y));
    }
}
static_assert(kNumParams % 2 == 0 && kOffWP0 % 2 == 0, "reduce_partials_kernel works on parameter pairs");

// ------------------------------------------------------------------------------------------
// loss gradient (train_network.py:54-55,85-89) and Adam (train_network.py:56,94)
// ------------------------------------------------------------------------------------------
__global__ void loss_grad_kernel(const float *__restrict__ policy, const float *__restrict__ value,
                                 const float *__restrict__ ptarget, const float *__restrict__ vtarget, int64_t B,
                                 float inv_total, float *__restrict__ loss, float *__restrict__ dpolicy,
                                 float *__restrict__ dvalue) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    aq_pdl_trigger();  // the heads backward that usually follows can load its weights while this grid drains
    float lp = 0.f, lv = 0.f;
    for (int64_t b = (int64_t)blockIdx.x * nwarps + warp; b < B; b += (int64_t)gridDim.x * nwarps) {
        // CrossEntropyLoss(input = softmax probabilities, target = probabilities):
        //   -sum_a t_a * log_softmax(p)_a   -- the second softmax is the reference's behaviour
        float p[7], t[7], mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < 7; ++k) {
            const int a = lane + 32 * k;
            p[k] = a < kP ? __ldg(policy + b * kP + a) : -INFINITY;
            t[k] = a < kP ? __ldg(ptarget + b * kP + a) : 0.f;
            mx = fmaxf(mx, p[k]);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
        float se = 0.f, tsum = 0.f;
#pragma unroll
        for (int k = 0; k < 7; ++k) {
            if (lane + 32 * k < kP) se += expf(p[k] - mx);
            tsum += t[k];
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            se += __shfl_xor_sync(0xffffffffu, se, d);
            tsum += __shfl_xor_sync(0xffffffffu, tsum, d);
        }
        const float lse = mx + logf(se);
        float l = 0.f;
#pragma unroll
        for (int k = 0; k < 7; ++k) {
            const int a = lane + 32 * k;
            if (a < kP) {
                const float ls = p[k] - lse;
                l -= t[k] * ls;
                dpolicy[b * kP + a] = (expf(ls) * tsum - t[k]) * inv_total;
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) l += __shfl_xor_sync(0xffffffffu, l, d);
        if (lane == 0) {
            const float dv = __ldg(value + b) - __ldg(vtarget + b);
            lp += l;
            lv += dv * dv;
            dvalue[b] = 2.f * dv * inv_total;
        }
    }
    // monitoring scalars only; gradients above do not depend on them.  One pair of atomics per CTA: a pair per warp
    // (4,096 warps on two addresses) serialised in L2 and cost 12 of the kernel's 16 us at B = 4096
    __shared__ float red[2][32];
    if (lane == 0) { red[0][warp] = lp; red[1][warp] = lv; }
    __syncthreads();
    if (warp == 0 && loss) {
        float a = lane < nwarps ? red[0][lane] : 0.f, c = lane < nwarps ? red[1][lane] : 0.f;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, d);
            c += __shfl_xor_sync(0xffffffffu, c, d);
        }
        if (lane == 0) {
            atomicAdd(loss + 0, a * inv_total);
            atomicAdd(loss + 1, c * inv_total);
        }
    }
}

__global__ void adam_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m,
                            float *__restrict__ v, int64_t n, float step_size, float bc2_sqrt, float beta1,
                            float beta2, float eps, float grad_scale) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float gi = g[i] * grad_scale;
    const float mi = m[i] + (1.f - beta1) * (gi - m[i]);        // exp_avg.lerp_(grad, 1 - beta1)
    const float vi = v[i] * beta2 + (1.f - beta2) * gi * gi;    // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;          // (exp_avg_sq.sqrt() / bias_correction2_sqrt).add_(eps)
    p[i] = p[i] - step_size * (mi / denom);
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" int64_t aq_gnn_backward_ws_floats(int64_t B) { return BwdWs{B}.total(); }

int aq_gcn_backward_tc2(const float *params, float *saved, const float *dg, int64_t B, float *partial, cudaStream_t st);  // gnn_tc2_bwd.cu

int aq_dp_adam_launch(void *comm, const float *grads_in, const float *partial, int gcn_slots, int head_slots, float *params, float *exp_avg,
                      float *exp_avg_sq, float *grads_out, float lr, float beta1, float beta2, float eps, bool pdl, cudaStream_t st);  // dp_comm.cu

#ifndef AQ_HEAD_CHUNK_ROWS
#define AQ_HEAD_CHUNK_ROWS 64
#endif
int aq_heads_wgrad_tc_slots(int64_t B);  // heads_wgrad_tc.cu
int aq_heads_wgrad_tc(const float *dhp, const float *dhv, const float *dz, const float *du, const float *pooled, const float *hp,
                      const float *hv, int64_t B, float *partial, cudaStream_t st);
// partial slots that hold head gradients: fp32 path (atb_jobs_kernel) one row chunk per 64 boards; tensor-core path one per 64-board tile
static inline int head_slot_count(int64_t B, int precision) {
    if (precision == 1) return aq_heads_wgrad_tc_slots(B);
    return (int)std::min<int64_t>(kSlots, (B + AQ_HEAD_CHUNK_ROWS - 1) / AQ_HEAD_CHUNK_ROWS);
}

// The backward kernels up to the partial-gradient slots.  Loss gradient either given (dpolicy, dvalue) or computed in the heads
// backward from the targets (ptarget, vtarget, B_total, loss).
static int backward_to_partials(const float *params, const float *saved, const float *dpolicy, const float *dvalue, const float *ptarget,
                                const float *vtarget, int64_t B, int64_t B_total, float *loss, float *workspace, int precision,
                                cudaStream_t st) {
    const SavedLayout L{B};
    const BwdWs W{B};
    const bool fused_loss = ptarget != nullptr;
    if (fused_loss && loss) {
        const cudaError_t e = cudaMemsetAsync(loss, 0, 2 * sizeof(float), st);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_loss_backward(memset)");
    }
    const int hb_threads = B <= 1184 ? 256 : kHbThreads;  // 148 CTAs x 8 boards cover 1,184 boards in one pass
    const int nb = B >= 8192 ? 4 : B >= kSlots * (kHbThreads / 32) ? 2 : 1;   // boards per warp at a time (HeadBwdSmem)
    const int64_t per_cta = (int64_t)(hb_threads / 32) * nb;
    const int64_t hb = (B + per_cta - 1) / per_cta;
    const dim3 hgrid((unsigned)(hb < kSlots ? hb : kSlots));
    const float inv_total = 1.0f / (float)(B_total > 0 ? B_total : B);
    // the backward kernels are chained by programmatic dependent launches: each reads only the parameters before its aq_pdl_wait()
    auto launch_hb = [&](auto kernel, size_t smem) {
        return aq_launch("heads_backward_kernel", kernel, hgrid, hb_threads, smem, st, true, params, saved, dpolicy, dvalue, ptarget, vtarget,
                         inv_total, loss, B, workspace);
    };
    int rc;
    if (fused_loss) {
        if (nb == 4) rc = launch_hb(heads_backward_kernel<true, 4>, sizeof(HeadBwdSmem<4>));
        else if (nb == 2) rc = launch_hb(heads_backward_kernel<true, 2>, sizeof(HeadBwdSmem<2>));
        else rc = launch_hb(heads_backward_kernel<true, 1>, sizeof(HeadBwdSmem<1>));
    } else {
        if (nb == 4) rc = launch_hb(heads_backward_kernel<false, 4>, sizeof(HeadBwdSmem<4>));
        else if (nb == 2) rc = launch_hb(heads_backward_kernel<false, 2>, sizeof(HeadBwdSmem<2>));
        else rc = launch_hb(heads_backward_kernel<false, 1>, sizeof(HeadBwdSmem<1>));
    }
    if (rc) return rc;
    if (precision == 1)  // tensor-core trunk backward: fills the GCN ranges of every partial slot itself
        rc = aq_gcn_backward_tc2(params, const_cast<float *>(saved), workspace + W.dg(), B, workspace + W.partial(), st);
    else
        rc = aq_launch("gcn_backward_kernel", gcn_backward_kernel, kSlots, kGcnThreads, sizeof(GcnBwdSmem), st, false, params, saved, B, workspace);
    if (rc) return rc;

    if (precision == 1)   // head weight gradients on the tensor cores (the trunk backward above filled the GCN ranges of the slots)
        return aq_heads_wgrad_tc(workspace + W.dhp(), workspace + W.dhv(), workspace + W.dz(), workspace + W.du(), saved + L.pooled(),
                                 saved + L.hp(), saved + L.hv(), B, workspace + W.partial(), st);
    AtbJobs jobs;
    int nj = 0;
    // head jobs: one row chunk per 64 boards (at most kSlots); node-level jobs: kSlots chunks
    const int head_slots = head_slot_count(B, precision);
    auto add = [&](const float *A, int lda, int M, const float *Bm, int ldb, int N, int64_t R, int off, int bias_off = -1) {
        jobs.job[nj++] = AtbJob{A, lda, M, Bm, ldb, N, R, off, R == B ? head_slots : kSlots, bias_off};
    };
    const int64_t RN = B * kV;
    if (precision != 1) {
        add(workspace + W.dy1(), kH, kH, saved + L.ax0(), kF, kF, RN, kOffW1);    // dW1 = dY1^T (A_hat X0)
        add(workspace + W.dz2(), kH, kH, saved + L.x(0), kH, kH, RN, kOffW2);     // dW2 = dZ2^T X1
        add(workspace + W.dz3(), kH, kH, saved + L.x(1), kH, kH, RN, kOffW3);     // dW3 = dZ3^T X2
    }
    // each head layer's bias gradient (column sums of the same A) rides on its weight job
    add(workspace + W.dhp(), kHH, kHH, saved + L.pooled(), kH, kH, B, kOffWP0, kOffBP0);
    add(workspace + W.dz(), kP, kP, saved + L.hp(), kHH, kHH, B, kOffWP2, kOffBP2);
    add(workspace + W.dhv(), kHH, kHH, saved + L.pooled(), kH, kH, B, kOffWV0, kOffBV0);
    add(workspace + W.du(), 1, 1, saved + L.hv(), kHH, kHH, B, kOffWV2, kOffBV2);
    jobs.n = nj;
    return aq_launch("atb_jobs_kernel", atb_jobs_kernel, dim3(precision != 1 ? kSlots : head_slots, kMaxMTiles, nj), 256, 0, st, true, jobs,
                     workspace + W.partial());
}

extern "C" int aq_gnn_backward(const float *params, const float *saved, const float *dpolicy, const float *dvalue,
                               int64_t B, float *grads, float *workspace, int precision, void *stream) {
    if (B <= 0 || !params || !saved || !dpolicy || !dvalue || !grads || !workspace)
        return aq_set_error(AQ_ERR_ARG, "aq_gnn_backward");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = backward_to_partials(params, saved, dpolicy, dvalue, nullptr, nullptr, B, B, nullptr, workspace, precision, st);
    if (rc) return rc;
    return aq_launch("reduce_partials_kernel", reduce_partials_kernel, (kNumParams / 2 + kRedPairs - 1) / kRedPairs, kRedPairs * 4, 0, st, true,
                     (const float *)(workspace + BwdWs{B}.partial()), grads, head_slot_count(B, precision));
}

// One training step behind the forward pass, as the reference's `loss = ...; optimizer.zero_grad(); loss.backward(); optimizer.step()`
// (train_network.py:85-94) under data parallelism: loss gradient + heads backward (one kernel), trunk backward, head weight
// gradients, then ONE kernel that reduces the partial slots, all-reduces the flat gradient over the ranks of `comm` (NVLink peer
// memory, dp_comm.cu) and applies Adam.  grads (may be NULL) receives the reduced gradient (sum over the ranks).
extern "C" int aq_train_backward_step(void *comm, float *params, const float *saved, const float *policy_target, const float *value_target,
                                      int64_t B, int64_t B_total, float *loss, float *grads, float *exp_avg, float *exp_avg_sq,
                                      float *workspace, int precision, float lr, float beta1, float beta2, float eps, void *stream) {
    if (B <= 0 || B_total < B || !comm || !params || !saved || !policy_target || !value_target || !exp_avg || !exp_avg_sq || !workspace)
        return aq_set_error(AQ_ERR_ARG, "aq_train_backward_step");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = backward_to_partials(params, saved, nullptr, nullptr, policy_target, value_target, B, B_total, loss, workspace, precision, st);
    if (rc) return rc;
    return aq_dp_adam_launch(comm, nullptr, workspace + BwdWs{B}.partial(), kSlots, head_slot_count(B, precision), params, exp_avg, exp_avg_sq, grads, lr,
                             beta1, beta2, eps, /*pdl=*/true, st);
}

extern "C" int aq_loss_grad(const float *policy, const float *value, const float *policy_target,
                            const float *value_target, int64_t B, int64_t B_total, float *loss, float *dpolicy,
                            float *dvalue, void *stream) {
    if (B <= 0 || B_total <= 0 || !policy || !value || !policy_target || !value_target || !dpolicy || !dvalue)
        return aq_set_error(AQ_ERR_ARG, "aq_loss_grad");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (loss) {
        cudaError_t e = cudaMemsetAsync(loss, 0, 2 * sizeof(float), st);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_loss_grad(memset)");
    }
    const int64_t nb = (B + 7) / 8;
    return aq_launch("loss_grad_kernel", loss_grad_kernel, (unsigned)(nb < 1184 ? nb : 1184), 256, 0, st, false, policy, value, policy_target,
                     value_target, B, 1.0f / (float)B_total, loss, dpolicy, dvalue);
}

extern "C" int aq_adam_step(float *params, const float *grads, float *exp_avg, float *exp_avg_sq, int64_t n,
                            int64_t step, float lr, float beta1, float beta2, float eps, float grad_scale,
                            void *stream) {
    if (n <= 0 || step <= 0 || !params || !grads || !exp_avg || !exp_avg_sq) return aq_set_error(AQ_ERR_ARG, "aq_adam_step");
    const double bc1 = 1.0 - pow((double)beta1, (double)step);
    const double bc2 = 1.0 - pow((double)beta2, (double)step);
    const float step_size = (float)((double)lr / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    return aq_launch("adam_kernel", adam_kernel, (unsigned)((n + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream), false, params,
                     grads, exp_avg, exp_avg_sq, n, step_size, bc2_sqrt, beta1, beta2, eps, grad_scale);
}
