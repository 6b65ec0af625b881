// GraphPolicyValueNetwork.forward (pv_network_gnn.py:53-64) -- fp32 FFMA path.
//   gcn_forward_fp32_kernel : graph build + 3 GCN layers + global_mean_pool, one board per CTA
//                             iteration, all activations resident in shared memory
//   heads_forward_kernel    : policy / value MLPs, softmax, tanh, optional legal-action
//                             renormalisation (BaseNetwork.predict semantics)
#include <cstdio>
#include <cstdlib>
#include <cuda_fp16.h>
#include "gnn_fp32.cuh"

using namespace aq;

// ------------------------------------------------------------------------------------------
// shared memory map of the GCN kernel (bytes): two weight tiles, two activation buffers
// (bufx's GEMM over-read of rows 81..87 lands in bufz / the small arrays, results discarded)
// ------------------------------------------------------------------------------------------
struct GcnSmem {
    float w2[kH * kH];
    float w3[kH * kH];
    float bufx[kV * kH];
    float bufz[kV * kH];
    float w1t[kF * kH];  // [f][n]   (w1t + b1..b3 = 1152 floats >= the 7x128 GEMM over-read of bufz)
    float b1[kH], b2[kH], b3[kH];
    float coef[kV * 5 + 3];
    float x0[kV * kF + 2];
    float ax0[kV * kF + 2];
    float red[256];
    uint8_t open_s[96];
};
static_assert(sizeof(GcnSmem) <= 227 * 1024, "GcnSmem exceeds the 227 KB shared memory limit");

template <bool kSave>
__global__ void __launch_bounds__(kGcnThreads, 1)
gcn_forward_fp32_kernel(const float *__restrict__ params, const AqState *__restrict__ states,
                        const float *__restrict__ x_in, const uint8_t *__restrict__ open_in, int64_t B,
                        float *__restrict__ pooled_out, float *__restrict__ saved) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    GcnSmem &sm = *reinterpret_cast<GcnSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // weights: W^T tiles so that the GEMM reads rows of the reduction index
    load_weight_transposed(sm.w2, params + kOffW2, tid);
    load_weight_transposed(sm.w3, params + kOffW3, tid);
    for (int i = tid; i < kF * kH; i += kGcnThreads) {
        const int n = i / kF, f = i % kF;
        sm.w1t[f * kH + n] = __ldg(params + kOffW1 + i);
    }
    if (tid < kH) {
        sm.b1[tid] = __ldg(params + kOffB1 + tid);
        sm.b2[tid] = __ldg(params + kOffB2 + tid);
        sm.b3[tid] = __ldg(params + kOffB3 + tid);
    }
    const SavedLayout L{B};

    for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
        __syncthreads();  // previous board fully consumed (also covers the weight fill)
        // ---- inputs: node features + open-direction masks --------------------------------
        if (states) {
            const AqState s = load_state(states + b);
            board_inputs_from_state(s, sm.x0, sm.open_s, tid);
        } else {
            for (int i = tid; i < kV * kF; i += kGcnThreads) sm.x0[i] = __ldg(x_in + b * kV * kF + i);
            if (tid < kV) sm.open_s[tid] = __ldg(open_in + b * kV + tid);
        }
        __syncthreads();
        board_coefficients(sm.open_s, sm.coef, tid);
        __syncthreads();
        // ---- layer 1: (A_hat X0) W1^T + b1, ReLU  (aggregate the 6-wide input first) -------
        for (int i = tid; i < kV * kF; i += kGcnThreads) {
            const int v = i / kF, f = i % kF;
            const float *c = sm.coef + v * 5;
            float s = c[0] * sm.x0[i];
            if (c[1] != 0.f) s = fmaf(c[1], sm.x0[(v - 9) * kF + f], s);
            if (c[2] != 0.f) s = fmaf(c[2], sm.x0[(v + 9) * kF + f], s);
            if (c[3] != 0.f) s = fmaf(c[3], sm.x0[(v - 1) * kF + f], s);
            if (c[4] != 0.f) s = fmaf(c[4], sm.x0[(v + 1) * kF + f], s);
            sm.ax0[i] = s;
        }
        __syncthreads();
        {
            const int n = tid & (kH - 1);
            float w[kF];
#pragma unroll
            for (int f = 0; f < kF; ++f) w[f] = sm.w1t[f * kH + n];
            const float bias = sm.b1[n];
            for (int v = tid >> 7; v < kV; v += 2) {
                float s = bias;
#pragma unroll
                for (int f = 0; f < kF; ++f) s = fmaf(sm.ax0[v * kF + f], w[f], s);
                sm.bufx[v * kH + n] = fmaxf(s, 0.f);
            }
        }
        __syncthreads();
        if (kSave) {
            float4 *dst = reinterpret_cast<float4 *>(saved + L.x(0) + b * kV * kH);
            const float4 *src = reinterpret_cast<const float4 *>(sm.bufx);
            for (int i = tid; i < kV * kH / 4; i += kGcnThreads) dst[i] = src[i];
            for (int i = tid; i < kV * 5; i += kGcnThreads) saved[L.coef() + b * kV * 5 + i] = sm.coef[i];
            for (int i = tid; i < kV * kF; i += kGcnThreads) saved[L.ax0() + b * kV * kF + i] = sm.ax0[i];
        }
        // ---- layers 2, 3: Z = X W^T ; X' = relu(A_hat Z + b) ----------------------------------
#pragma unroll 1
        for (int layer = 1; layer < kLayers; ++layer) {
            const float *wt = layer == 1 ? sm.w2 : sm.w3;
            const float *bias = layer == 1 ? sm.b2 : sm.b3;
            float acc[kRowsPerWarp][4];
            gemm_rows(sm.bufx, wt, warp, lane, acc);
#pragma unroll
            for (int i = 0; i < kRowsPerWarp; ++i) {
                const int r = warp * kRowsPerWarp + i;
                if (r < kV)
                    reinterpret_cast<float4 *>(sm.bufz)[r * 32 + lane] = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
            }
            __syncthreads();
            aggregate<true>(sm.bufz, sm.bufx, sm.coef, bias, warp, lane);
            __syncthreads();
            if (kSave) {
                float4 *dst = reinterpret_cast<float4 *>(saved + L.x(layer) + b * kV * kH);
                const float4 *src = reinterpret_cast<const float4 *>(sm.bufx);
                for (int i = tid; i < kV * kH / 4; i += kGcnThreads) dst[i] = src[i];
            }
        }
        // ---- global_mean_pool: every graph has exactly 81 nodes --------------------------------
        {
            const int n = tid & (kH - 1), half = tid >> 7;
            float s = 0.f;
            for (int v = half; v < kV; v += 2) s += sm.bufx[v * kH + n];
            sm.red[tid] = s;
        }
        __syncthreads();
        if (tid < kH) {
            const float g = (sm.red[tid] + sm.red[tid + kH]) / (float)kV;
            pooled_out[b * kH + tid] = g;
        }
    }
}

// ------------------------------------------------------------------------------------------
// heads: one warp per board; weights transposed in shared memory ([k][j], j fastest)
// ------------------------------------------------------------------------------------------
constexpr int kHeadThreads = 256;
constexpr int kPPad = 224;  // 209 logits -> 7 per lane

struct HeadSmem {
    float wp0t[kH * kHH];     // [k][j]
    float wv0t[kH * kHH];
    float wp2t[kHH * kPPad];  // [j][a]
    float bp0[kHH], bv0[kHH], wv2[kHH];
    float bp2[kPPad];
    float g[kHeadThreads / 32][kH];
    float hp[kHeadThreads / 32][kHH];
    float hv[kHeadThreads / 32][kHH];
};
static_assert(sizeof(HeadSmem) <= 227 * 1024, "HeadSmem too large");

// mode 0: policy/value outputs (network forward). mode 1: predict semantics -- restrict to the
// legal mask and renormalise (pv_network_cnn.py:129-132).
template <bool kSave, bool kLegal>
__global__ void __launch_bounds__(kHeadThreads, 1)
heads_forward_kernel(const float *__restrict__ params, const float *__restrict__ pooled, int64_t B,
                     float *__restrict__ policy, float *__restrict__ value, const uint32_t *__restrict__ mask,
                     float *__restrict__ saved) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    HeadSmem &sm = *reinterpret_cast<HeadSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < kHH * kH; i += kHeadThreads) {
        const int j = i >> 7, k = i & 127;
        sm.wp0t[k * kHH + j] = __ldg(params + kOffWP0 + i);
        sm.wv0t[k * kHH + j] = __ldg(params + kOffWV0 + i);
    }
    for (int i = tid; i < kHH * kPPad; i += kHeadThreads) {
        const int j = i / kPPad, a = i % kPPad;
        sm.wp2t[i] = a < kP ? __ldg(params + kOffWP2 + a * kHH + j) : 0.f;
    }
    if (tid < kHH) {
        sm.bp0[tid] = __ldg(params + kOffBP0 + tid);
        sm.bv0[tid] = __ldg(params + kOffBV0 + tid);
        sm.wv2[tid] = __ldg(params + kOffWV2 + tid);
    }
    if (tid < kPPad) sm.bp2[tid] = tid < kP ? __ldg(params + kOffBP2 + tid) : 0.f;
    const float bv2 = __ldg(params + kOffBV2);
    __syncthreads();
    const SavedLayout L{B};
    const int nwarps = kHeadThreads / 32;

    for (int64_t b = (int64_t)blockIdx.x * nwarps + warp; b < B; b += (int64_t)gridDim.x * nwarps) {
        __syncwarp();
        reinterpret_cast<float4 *>(sm.g[warp])[lane] = __ldg(reinterpret_cast<const float4 *>(pooled + b * kH) + lane);
        __syncwarp();
        // hidden layers of both heads: outputs j = lane, lane+32
        float p0 = sm.bp0[lane], p1 = sm.bp0[lane + 32], v0 = sm.bv0[lane], v1 = sm.bv0[lane + 32];
#pragma unroll 4
        for (int k = 0; k < kH; ++k) {
            const float gk = sm.g[warp][k];
            p0 = fmaf(gk, sm.wp0t[k * kHH + lane], p0);
            p1 = fmaf(gk, sm.wp0t[k * kHH + lane + 32], p1);
            v0 = fmaf(gk, sm.wv0t[k * kHH + lane], v0);
            v1 = fmaf(gk, sm.wv0t[k * kHH + lane + 32], v1);
        }
        p0 = fmaxf(p0, 0.f); p1 = fmaxf(p1, 0.f); v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f);
        sm.hp[warp][lane] = p0; sm.hp[warp][lane + 32] = p1;
        sm.hv[warp][lane] = v0; sm.hv[warp][lane + 32] = v1;
        if (kSave) {
            saved[L.hp() + b * kHH + lane] = p0; saved[L.hp() + b * kHH + lane + 32] = p1;
            saved[L.hv() + b * kHH + lane] = v0; saved[L.hv() + b * kHH + lane + 32] = v1;
        }
        __syncwarp();
        // value: Linear(64 -> 1) + tanh
        float u = v0 * sm.wv2[lane] + v1 * sm.wv2[lane + 32];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) u += __shfl_xor_sync(0xffffffffu, u, d);
        const float val = tanhf(u + bv2);
        // policy logits a = lane + 32 t
        float z[7];
#pragma unroll
        for (int t = 0; t < 7; ++t) z[t] = sm.bp2[lane + 32 * t];
#pragma unroll 2
        for (int j = 0; j < kHH; ++j) {
            const float h = sm.hp[warp][j];
#pragma unroll
            for (int t = 0; t < 7; ++t) z[t] = fmaf(h, sm.wp2t[j * kPPad + lane + 32 * t], z[t]);
        }
        float mx = -INFINITY;
#pragma unroll
        for (int t = 0; t < 7; ++t) if (lane + 32 * t < kP) mx = fmaxf(mx, z[t]);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
        float sum = 0.f;
#pragma unroll
        for (int t = 0; t < 7; ++t) {
            z[t] = (lane + 32 * t < kP) ? expf(z[t] - mx) : 0.f;
            sum += z[t];
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
#pragma unroll
        for (int t = 0; t < 7; ++t) z[t] = z[t] / sum;  // softmax probabilities
        if (kSave) {
#pragma unroll
            for (int t = 0; t < 7; ++t) if (lane + 32 * t < kP) saved[L.policy() + b * kP + lane + 32 * t] = z[t];
            if (lane == 0) saved[L.value() + b] = val;
        }
        if (kLegal) {
            // policy = policy[legal]; policy /= sum(policy) if sum(policy) else 1
            float ls = 0.f;
#pragma unroll
            for (int t = 0; t < 7; ++t) {
                const bool legal = (__ldg(mask + b * 8 + t) >> lane) & 1;  // word t holds actions 32t..32t+31
                z[t] = legal ? z[t] : 0.f;
                ls += z[t];
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) ls += __shfl_xor_sync(0xffffffffu, ls, d);
            if (ls != 0.f) {
#pragma unroll
                for (int t = 0; t < 7; ++t) z[t] = z[t] / ls;
            }
        }
#pragma unroll
        for (int t = 0; t < 7; ++t) if (lane + 32 * t < kP) policy[b * kP + lane + 32 * t] = z[t];
        if (lane == 0) value[b] = val;
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
int aq_gcn_forward_tc2(const float *params, const void *prepared, const AqState *states, int64_t B, float *pooled, float *saved,
                       uint32_t *mask, uint8_t *pawn, bool after_legal, cudaStream_t st);  // gnn_tc2.cu
int aq_heads_forward_tc(const float *params, const void *prepared, const float *pooled, int64_t B, float *policy, float *value,
                        const uint32_t *legal_mask, float *saved, bool pdl, cudaStream_t st);  // heads_tc.cu

static int launch_trunk(const float *params, const void *prepared, const AqState *states, const float *x,
                        const uint8_t *open_mask, int64_t B, float *pooled, float *saved, int precision, cudaStream_t st,
                        bool after_legal = false, uint32_t *legal_out = nullptr, uint8_t *pawn_out = nullptr) {
    if (precision == 1) {
        if (!states) return aq_set_error(AQ_ERR_UNSUPPORTED, "aq_gnn_forward(bf16 path needs packed states)");
        return aq_gcn_forward_tc2(params, prepared, states, B, pooled, saved, saved ? nullptr : legal_out, pawn_out, saved ? false : after_legal, st);
    }
    const unsigned grid = (unsigned)(B < aq_num_sms() ? B : aq_num_sms());
    if (saved)
        return aq_launch("gcn_forward_fp32_kernel", gcn_forward_fp32_kernel<true>, grid, kGcnThreads, sizeof(GcnSmem), st, false, params, states,
                         x, open_mask, B, pooled, saved);
    return aq_launch("gcn_forward_fp32_kernel", gcn_forward_fp32_kernel<false>, grid, kGcnThreads, sizeof(GcnSmem), st, false, params, states,
                     x, open_mask, B, pooled, (float *)nullptr);
}

static int launch_heads(const float *params, const void *prepared, const float *pooled, int64_t B, float *policy,
                        float *value, const uint32_t *legal_mask, float *saved, int precision, cudaStream_t st, bool after_trunk = false) {
    // tensor-core heads: inference, and the training forward (hidden activations etc. saved by the kernel).  (Measured at B = 256: the
    // warp-per-board kernel is no faster there -- 26 us against 23 us: its 116 KB weight fill per CTA costs what the tile chain costs.)
    if (precision == 1 && (!saved || !legal_mask))
        return aq_heads_forward_tc(params, prepared, pooled, B, policy, value, legal_mask, saved, after_trunk, st);
    const int64_t hb = (B + 7) / 8;
    const unsigned hgrid = (unsigned)(hb < aq_num_sms() ? hb : aq_num_sms());
    if (legal_mask)
        return aq_launch("heads_forward_kernel", heads_forward_kernel<false, true>, hgrid, kHeadThreads, sizeof(HeadSmem), st, false, params,
                         pooled, B, policy, value, legal_mask, (float *)nullptr);
    if (saved)
        return aq_launch("heads_forward_kernel", heads_forward_kernel<true, false>, hgrid, kHeadThreads, sizeof(HeadSmem), st, false, params,
                         pooled, B, policy, value, (const uint32_t *)nullptr, saved);
    return aq_launch("heads_forward_kernel", heads_forward_kernel<false, false>, hgrid, kHeadThreads, sizeof(HeadSmem), st, false, params,
                     pooled, B, policy, value, (const uint32_t *)nullptr, (float *)nullptr);
}

extern "C" int aq_gcn_trunk_forward(const float *params, const void *prepared, const AqState *states, int64_t B,
                                    float *pooled, int precision, void *stream) {
    if (B < 0 || !params || (B > 0 && (!states || !pooled))) return aq_set_error(AQ_ERR_ARG, "aq_gcn_trunk_forward");
    if (B == 0) return 0;
    return launch_trunk(params, prepared, states, nullptr, nullptr, B, pooled, nullptr, precision, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int aq_heads_forward(const float *params, const void *prepared, const float *pooled, int64_t B, float *policy,
                                float *value, const uint32_t *legal_mask, int precision, void *stream) {
    if (B < 0 || !params || (B > 0 && (!pooled || !policy || !value))) return aq_set_error(AQ_ERR_ARG, "aq_heads_forward");
    if (B == 0) return 0;
    return launch_heads(params, prepared, pooled, B, policy, value, legal_mask, nullptr, precision, reinterpret_cast<cudaStream_t>(stream));
}

// pooled [B,128] scratch must be provided by the caller when saved == NULL (inference); with a
// saved workspace the pooled section of `saved` is used.
// legal_out != nullptr (precision 1 inference): the trunk launch also writes legal_mask = legal_out and pawn_out (aq_leaf_eval).
int aq_gnn_forward_impl(const float *params, const void *prepared, const AqState *states, const float *x,
                        const uint8_t *open_mask, int64_t B, float *policy, float *value, float *saved, float *pooled_scratch,
                        const uint32_t *legal_mask, int precision, cudaStream_t st, bool after_legal = false,
                        uint32_t *legal_out = nullptr, uint8_t *pawn_out = nullptr) {
    if (B == 0) return 0;
    const SavedLayout L{B};
    float *pooled = saved ? saved + L.pooled() : pooled_scratch;
    if (!pooled) return aq_set_error(AQ_ERR_ARG, "aq_gnn_forward(pooled scratch)");
    int rc = launch_trunk(params, prepared, states, x, open_mask, B, pooled, saved, precision, st, after_legal, legal_out, pawn_out);
    if (rc) return rc;
    return launch_heads(params, prepared, pooled, B, policy, value, legal_mask, saved, precision, st, /*after_trunk=*/true);
}

extern "C" int64_t aq_param_count(void) { return kNumParams; }
extern "C" int64_t aq_gnn_saved_floats(int64_t B) { return SavedLayout{B}.total(); }

extern "C" int aq_gnn_forward(const float *params, const AqState *states, const float *x, const uint8_t *open_mask,
                              int64_t B, float *policy, float *value, float *saved, int precision, void *stream) {
    if (B < 0 || !params || (B > 0 && (!policy || !value)) || (B > 0 && !states && (!x || !open_mask)))
        return aq_set_error(AQ_ERR_ARG, "aq_gnn_forward");
    if (B == 0) return 0;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    // inference without a saved workspace: the pooled [B,128] vector needs scratch; take it from the
    // stream-ordered pool (no persistent allocation, freed on the same stream)
    float *scratch = nullptr;
    if (!saved) {
        cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&scratch), (size_t)B * kH * sizeof(float), st);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_gnn_forward(cudaMallocAsync)");
    }
    int rc = aq_gnn_forward_impl(params, nullptr, states, x, open_mask, B, policy, value, saved, scratch, nullptr, precision, st);
    if (scratch) cudaFreeAsync(scratch, st);
    return rc;
}

// workspace of one leaf evaluation: pooled [B,128] | the legal-mask task list (aq_legal_mask_ws_bytes; used by the fp32 path, the bf16
// path computes the mask inside the trunk launch with a task list in shared memory)
extern "C" int64_t aq_legal_mask_ws_bytes(int64_t B);
extern "C" int aq_legal_mask_ws(const AqState *states, int64_t B, uint32_t *mask, uint8_t *pawn, void *ws, int64_t ws_bytes, void *stream);
constexpr int64_t kLeafFusedMin = 4096;
static inline int64_t leaf_pooled_floats(int64_t B) { return (B * kH + 63) / 64 * 64; }
extern "C" int64_t aq_leaf_eval_ws_floats(int64_t B) { return leaf_pooled_floats(B) + (aq_legal_mask_ws_bytes(B) + 3) / 4; }

extern "C" int aq_leaf_eval(const float *params, const void *prepared, const AqState *states, int64_t B, float *priors,
                            float *value, uint32_t *mask, uint8_t *pawn, float *workspace, int precision, void *stream) {
    if (B < 0 || !params || (B > 0 && (!states || !priors || !value || !mask || !pawn || !workspace)))
        return aq_set_error(AQ_ERR_ARG, "aq_leaf_eval");
    if (B == 0) return 0;
    const cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    // precision 1 from kLeafFusedMin boards: one launch computes the trunk and, in a fifth warpgroup of each CTA, the legal mask; then
    // the heads.  Below, a CTA has too few boards to hide the mask's dependency chain under them (B200: 256 boards 27.5 us unfused,
    // 33.8 us fused; 4,096: 74.8 / 63.4 us): the legal-mask kernels run first and the trunk is launched programmatically behind them.
    if (precision == 1 && B >= kLeafFusedMin)
        return aq_gnn_forward_impl(params, prepared, states, nullptr, nullptr, B, priors, value, nullptr, workspace, mask, precision, st,
                                   false, mask, pawn);
    int rc = aq_legal_mask_ws(states, B, mask, pawn, workspace + leaf_pooled_floats(B), aq_legal_mask_ws_bytes(B), stream);
    if (rc) return rc;
    // the trunk does not read the legal mask: it is launched programmatically behind the legal-mask kernel (see aq_gcn_forward_tc2)
    return aq_gnn_forward_impl(params, prepared, states, nullptr, nullptr, B, priors, value, nullptr, workspace, mask, precision, st,
                               /*after_legal=*/true);
}

// ---- host-buffer variant ----------------------------------------------------------------------
// device workspace layout: states | priors | value | mask | pawn | pooled
static inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// every chunk of the pipelined host path owns a leaf-evaluation workspace for its `per` boards; the workspace size is linear
// in the board count plus a constant < 32 KB, so all chunks together fit host_ws_region_bytes(B)
constexpr int kHostMaxChunks = 8;
static inline size_t host_chunk_ws_bytes(int64_t per) { return align256((size_t)aq_leaf_eval_ws_floats(per) * 4); }
static inline size_t host_ws_region_bytes(int64_t B) {
    const size_t saturated = B > ((int64_t)1 << 23) ? kHostMaxChunks * (size_t)aq_legal_mask_ws_bytes(B) : 0;  // the task list stops growing at 2^23 states
    return host_chunk_ws_bytes(B + 128 * kHostMaxChunks) + kHostMaxChunks * (size_t)32768 + saturated;
}

extern "C" int64_t aq_leaf_eval_host_ws_bytes(int64_t B) {
    return (int64_t)(align256((size_t)B * sizeof(AqState)) + align256((size_t)B * kP * 4) + align256((size_t)B * 4) +
                     align256((size_t)B * 32) + align256((size_t)B * 8) + host_ws_region_bytes(B));
}

// Host-side context for the pipelined host-buffer path: worker streams, their events, and a small cache of
// instantiated CUDA graphs (one per distinct argument tuple).  Owned by the caller (aq_host_ctx_create /
// aq_host_ctx_destroy); no global state.
struct AqHostKey {
    const void *params, *prepared, *states_host, *priors_host, *value_host, *mask_host, *pawn_host, *dev_ws;
    int64_t B;
    int precision;
    bool operator==(const AqHostKey &o) const {
        return params == o.params && prepared == o.prepared && states_host == o.states_host && priors_host == o.priors_host &&
               value_host == o.value_host && mask_host == o.mask_host && pawn_host == o.pawn_host && dev_ws == o.dev_ws &&
               B == o.B && precision == o.precision;
    }
};
constexpr int kHostGraphSlots = 8;
struct AqHostPending {  // a batch between aq_leaf_eval_host_compact_submit and _wait
    bool active = false;
    int64_t B = 0, priors_capacity = 0, copied = 0;
    int elem = 4;  // bytes per ragged prior on the wire
    void *priors_host = nullptr;
    unsigned char *d_compact = nullptr;
    int32_t *offsets_host = nullptr;
    cudaStream_t origin = nullptr;
};
struct AqHostCtx {
    cudaStream_t s[2];
    cudaEvent_t ready, done[2], chunk_done[8];
    AqHostPending pending;
    AqHostKey key[kHostGraphSlots];
    cudaGraphExec_t exec[kHostGraphSlots];
    int n_graphs, next_slot;
    int64_t est_per_board_x1024 = 0;  // running estimate of legal actions per board (x1024) that sizes the ragged priors copy; 0 = none yet
    int64_t short_copies = 0;         // batches that needed a second copy
};

extern "C" int aq_host_ctx_create(void **ctx) {
    if (!ctx) return aq_set_error(AQ_ERR_ARG, "aq_host_ctx_create");
    AqHostCtx *c = new AqHostCtx();
    c->n_graphs = c->next_slot = 0;
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaStreamCreateWithFlags(&c->s[i], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ready, cudaEventDisableTiming);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&c->done[i], cudaEventDisableTiming);
    for (int i = 0; i < 8 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&c->chunk_done[i], cudaEventDisableTiming);
    if (e != cudaSuccess) { delete c; return aq_set_error((int)e, "aq_host_ctx_create"); }
    *ctx = c;
    return 0;
}

extern "C" int aq_host_ctx_destroy(void *ctx) {
    if (!ctx) return 0;
    AqHostCtx *c = reinterpret_cast<AqHostCtx *>(ctx);
    for (int i = 0; i < c->n_graphs; ++i) cudaGraphExecDestroy(c->exec[i]);
    for (int i = 0; i < 2; ++i) { cudaStreamDestroy(c->s[i]); cudaEventDestroy(c->done[i]); }
    for (int i = 0; i < 8; ++i) cudaEventDestroy(c->chunk_done[i]);
    cudaEventDestroy(c->ready);
    delete c;
    return 0;
}

// Enqueues H2D -> leaf evaluation -> D2H for B states in `nchunk` chunks.  nchunk == 1: everything in order on
// `origin`.  nchunk > 1: chunks alternate between the two worker streams (forked from / joined back into
// `origin`), so the D2H of one chunk overlaps the kernels of the next.  Works eagerly and under stream capture.
static int enqueue_host_pipeline(AqHostCtx *ctx, cudaStream_t origin, int nchunk, const AqHostKey &k) {
    const int64_t B = k.B;
    unsigned char *p = reinterpret_cast<unsigned char *>(const_cast<void *>(k.dev_ws));
    AqState *d_states = reinterpret_cast<AqState *>(p); p += align256((size_t)B * sizeof(AqState));
    float *d_priors = reinterpret_cast<float *>(p);     p += align256((size_t)B * kP * 4);
    float *d_value = reinterpret_cast<float *>(p);      p += align256((size_t)B * 4);
    uint32_t *d_mask = reinterpret_cast<uint32_t *>(p); p += align256((size_t)B * 32);
    uint8_t *d_pawn = reinterpret_cast<uint8_t *>(p);   p += align256((size_t)B * 8);
    unsigned char *d_chunk_ws = p;
    const AqState *states_host = reinterpret_cast<const AqState *>(k.states_host);
    float *priors_host = reinterpret_cast<float *>(const_cast<void *>(k.priors_host));
    float *value_host = reinterpret_cast<float *>(const_cast<void *>(k.value_host));
    uint32_t *mask_host = reinterpret_cast<uint32_t *>(const_cast<void *>(k.mask_host));
    uint8_t *pawn_host = reinterpret_cast<uint8_t *>(const_cast<void *>(k.pawn_host));
    cudaError_t e = cudaSuccess;
    if (nchunk > 1) {
        e = cudaEventRecord(ctx->ready, origin);
        for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaStreamWaitEvent(ctx->s[i], ctx->ready, 0);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_leaf_eval_host(fork)");
    }
    // chunk boundaries are multiples of 128 boards (the heads kernel works on tiles of 128)
    const int64_t per = ((B + nchunk - 1) / nchunk + 127) / 128 * 128;
    for (int c = 0; c < nchunk; ++c) {
        const int64_t lo = (int64_t)c * per, n = (lo + per <= B ? per : B - lo);
        if (n <= 0) break;
        cudaStream_t cs = nchunk > 1 ? ctx->s[c & 1] : origin;
        e = cudaMemcpyAsync(d_states + lo, states_host + lo, (size_t)n * sizeof(AqState), cudaMemcpyHostToDevice, cs);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_leaf_eval_host(H2D)");
        int rc = aq_leaf_eval(reinterpret_cast<const float *>(k.params), k.prepared, d_states + lo, n, d_priors + lo * kP,
                              d_value + lo, d_mask + lo * 8, d_pawn + lo * 8,
                              reinterpret_cast<float *>(d_chunk_ws + (size_t)c * host_chunk_ws_bytes(per)), k.precision, cs);
        if (rc) return rc;
        e = cudaMemcpyAsync(priors_host + lo * kP, d_priors + lo * kP, (size_t)n * kP * 4, cudaMemcpyDeviceToHost, cs);
        if (e == cudaSuccess) e = cudaMemcpyAsync(value_host + lo, d_value + lo, (size_t)n * 4, cudaMemcpyDeviceToHost, cs);
        if (e == cudaSuccess && mask_host) e = cudaMemcpyAsync(mask_host + lo * 8, d_mask + lo * 8, (size_t)n * 32, cudaMemcpyDeviceToHost, cs);
        if (e == cudaSuccess && pawn_host) e = cudaMemcpyAsync(pawn_host + lo * 8, d_pawn + lo * 8, (size_t)n * 8, cudaMemcpyDeviceToHost, cs);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_leaf_eval_host(D2H)");
    }
    if (nchunk > 1) {
        for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
            e = cudaEventRecord(ctx->done[i], ctx->s[i]);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(origin, ctx->done[i], 0);
        }
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_leaf_eval_host(join)");
    }
    return 0;
}

static bool is_pinned_host(const void *ptr) {
    if (!ptr) return true;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// Looks up / builds the instantiated graph of the pipeline for this argument tuple.  The pipeline is captured on
// the context's own stream (the caller's stream may be the legacy default stream, which cannot be captured).
static cudaGraphExec_t host_graph_for(AqHostCtx *ctx, int nchunk, const AqHostKey &k) {
    for (int i = 0; i < ctx->n_graphs; ++i)
        if (ctx->key[i] == k) return ctx->exec[i];
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    if (cudaStreamBeginCapture(ctx->s[0], cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    // inside the capture s[0] is the origin and also one of the two workers: the fork/join events keep the order
    const int rc = enqueue_host_pipeline(ctx, ctx->s[0], nchunk, k);
    const cudaError_t e = cudaStreamEndCapture(ctx->s[0], &graph);
    if (rc != 0 || e != cudaSuccess || !graph) { cudaGetLastError(); if (graph) cudaGraphDestroy(graph); return nullptr; }
    if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) { cudaGetLastError(); exec = nullptr; }
    cudaGraphDestroy(graph);
    if (!exec) return nullptr;
    int slot;
    if (ctx->n_graphs < kHostGraphSlots) slot = ctx->n_graphs++;
    else { slot = ctx->next_slot; ctx->next_slot = (ctx->next_slot + 1) % kHostGraphSlots; cudaGraphExecDestroy(ctx->exec[slot]); }
    ctx->key[slot] = k;
    ctx->exec[slot] = exec;
    return exec;
}

extern "C" int aq_leaf_eval_host(const float *params, const void *prepared, const AqState *states_host, int64_t B, float *priors_host,
                                 float *value_host, uint32_t *mask_host, uint8_t *pawn_host, void *dev_ws,
                                 int precision, void *host_ctx, void *stream) {
    if (B < 0 || !params || (B > 0 && (!states_host || !priors_host || !value_host || !dev_ws)))
        return aq_set_error(AQ_ERR_ARG, "aq_leaf_eval_host");
    if (B == 0) return 0;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    AqHostCtx *ctx = reinterpret_cast<AqHostCtx *>(host_ctx);
    const AqHostKey k{params, prepared, states_host, priors_host, value_host, mask_host, pawn_host, dev_ws, B, precision};
    // with a context, batches >= 4096 are split in two so that the D2H of the first half overlaps the kernels of the second; when all
    // host buffers are pinned the whole pipeline is one CUDA graph per argument tuple (~40 API calls -> one launch)
    const int nchunk = (ctx && B >= 4096) ? 2 : 1;  // measured: 2 chunks beat 1, 3, 4 and 6 at B = 16384
    cudaError_t e = cudaSuccess;
    cudaGraphExec_t exec = nullptr;
    if (ctx && is_pinned_host(states_host) && is_pinned_host(priors_host) && is_pinned_host(value_host) &&
        is_pinned_host(mask_host) && is_pinned_host(pawn_host))
        exec = host_graph_for(ctx, nchunk, k);
    if (exec) {
        e = cudaGraphLaunch(exec, st);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_leaf_eval_host(graph launch)");
    } else {
        const int rc = enqueue_host_pipeline(ctx, st, nchunk, k);
        if (rc) return rc;
    }
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return aq_set_error((int)e, "aq_leaf_eval_host(sync)");
    return 0;
}

// ---- predict()-shaped output: priors of the LEGAL actions only, in legal_actions() order ----------------
// BaseNetwork.predict (BaseNetwork.py:36-40; pv_network_cnn.py:128-135) returns, per state, the probabilities of the
// legal actions only, ordered like state.legal_actions().  For a batch that is a ragged array: board b owns
// compact[offsets[b] .. offsets[b+1]).  Moving this form to the host instead of the dense [B,209] matrix is what the
// host-buffer path is bound by (PCIe): 4 bytes per legal action instead of 836 per board.

// offsets[b] = number of legal actions of boards < b (exclusive scan of popcount(mask)), offsets[B] = total.
// One CTA; thread t owns the contiguous run of ceil(B / 1024) boards starting at t * run: all of a thread's mask loads are issued
// before the first use (a tile-by-tile scan with two block barriers per 1,024 boards paid the load latency 16 times at B = 16,384),
// one block-wide scan of the 1,024 run totals, then every thread writes its run.  B is at most a few 10^4 per call on this path;
// runs longer than kScanRun are walked in pieces with a running carry.
constexpr int kScanRun = 16;
__global__ void __launch_bounds__(1024)
legal_count_scan_kernel(const uint32_t *mask, int64_t B, int32_t *__restrict__ offsets) {
    __shared__ int warp_sum[32];
    __shared__ int carry_s;
    aq_pdl_trigger();  // the compaction kernel behind this one may be scheduled; it waits for this grid before it reads the offsets
    aq_pdl_wait();  // launched programmatically behind the kernels that finalise the mask (coherent loads below: PDL rule, aq_common.cuh)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (int64_t base = 0; base < B; base += 1024 * kScanRun) {
        const int64_t left = B - base;
        const int run = (int)((left < 1024 * kScanRun ? left : 1024 * kScanRun) + 1023) / 1024;  // boards per thread in this piece
        const int64_t b0 = base + (int64_t)tid * run;
        int c[kScanRun];
#pragma unroll
        for (int k = 0; k < kScanRun; ++k) {
            c[k] = 0;
            if (k < run && b0 + k < B) {
                const uint4 lo = __ldcg(reinterpret_cast<const uint4 *>(mask + 8 * (b0 + k)));
                const uint4 hi = __ldcg(reinterpret_cast<const uint4 *>(mask + 8 * (b0 + k)) + 1);
                c[k] = __popc(lo.x) + __popc(lo.y) + __popc(lo.z) + __popc(lo.w) + __popc(hi.x) + __popc(hi.y) + __popc(hi.z) + __popc(hi.w);
            }
        }
        int mine = 0;
#pragma unroll
        for (int k = 0; k < kScanRun; ++k) mine += c[k];
        int incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = warp_sum[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, w, d);
                if (lane >= d) w += t;
            }
            warp_sum[lane] = w;  // inclusive scan of the warp totals
        }
        __syncthreads();
        const int carry = carry_s;
        int at = carry + (warp ? warp_sum[warp - 1] : 0) + incl - mine;
#pragma unroll
        for (int k = 0; k < kScanRun; ++k)
            if (k < run && b0 + k < B) { offsets[b0 + k] = at; at += c[k]; }
        __syncthreads();
        if (tid == 1023) carry_s = carry + warp_sum[31];
        __syncthreads();
    }
    if (tid == 0) offsets[B] = carry_s;
}

// One warp per board: every legal action's probability goes to its rank in legal_actions() order
// (pawn list order, then per wall slot H before V -- game_logic.py:103-117, 350-357).
// T = float (the bits of the dense priors) or __half (16-bit wire format of the host path, round to nearest even).
template <typename T>
__global__ void __launch_bounds__(256)
compact_priors_kernel(const float *priors, const uint32_t *mask, const uint8_t *pawn, const int32_t *offsets, int64_t B,
                      T *__restrict__ compact) {
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    aq_pdl_wait();  // launched programmatically behind the scan (and, through it, the heads kernel): coherent loads below
    if (b >= B) return;
    const uint32_t *m = mask + 8 * b;
    const uint32_t mw = lane < 8 ? __ldcg(m + lane) : 0u;
    uint32_t w[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) w[k] = __shfl_sync(0xffffffffu, mw, k);
    // wall bits: H = actions 81..144, V = actions 145..208
    const u64 lo2 = ((u64)w[3] << 32) | w[2], hi2 = ((u64)w[5] << 32) | w[4], top = ((u64)w[7] << 32) | w[6];
    const u64 legalH = (lo2 >> 17) | (hi2 << 47);            // bit s = action 81 + s
    const u64 legalV = (hi2 >> 17) | (top << 47);            // bit s = action 145 + s
    const uint2 pw = __ldcg(reinterpret_cast<const uint2 *>(pawn + 8 * b));
    const int np = pw.x & 0xFF;
    T *out = compact + __ldcg(offsets + b);
    const float *p = priors + (int64_t)kP * b;
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        const int a = lane + 32 * k;
        if (a >= kP || !((w[a >> 5] >> (a & 31)) & 1)) continue;
        int rank;
        if (a < AQ_SQUARES) {
            const u64 list = ((u64)pw.y << 32 | pw.x) >> 8;  // p0..p4
            rank = 0;
#pragma unroll
            for (int j = 0; j < 5; ++j)
                if (j < np && (int)((list >> (8 * j)) & 0xFF) == a) rank = j;
        } else {
            const bool isV = a >= AQ_SQUARES + AQ_SLOTS;
            const int slot = a - AQ_SQUARES - (isV ? AQ_SLOTS : 0);
            const u64 below = (1ull << slot) - 1ull;
            rank = np + __popcll(legalH & below) + __popcll(legalV & below) + (isV ? (int)((legalH >> slot) & 1) : 0);
        }
        if constexpr (sizeof(T) == 4) out[rank] = __ldcg(p + a);
        else out[rank] = __float2half_rn(__ldcg(p + a));
    }
}

static int compact_priors_impl(const float *priors, const uint32_t *mask, const uint8_t *pawn, int64_t B, int32_t *offsets, void *compact,
                               int wire, cudaStream_t st) {
    const int rc = aq_launch("aq_compact_priors(scan)", legal_count_scan_kernel, 1, 1024, 0, st, true, mask, B, offsets);
    if (rc || B == 0) return rc;
    const unsigned grid = (unsigned)((B + 7) / 8);
    if (wire == AQ_WIRE_F16)
        return aq_launch("aq_compact_priors", compact_priors_kernel<__half>, grid, 256, 0, st, true, priors, mask, pawn, (const int32_t *)offsets,
                         B, reinterpret_cast<__half *>(compact));
    return aq_launch("aq_compact_priors", compact_priors_kernel<float>, grid, 256, 0, st, true, priors, mask, pawn, (const int32_t *)offsets, B,
                     reinterpret_cast<float *>(compact));
}

extern "C" int aq_compact_priors(const float *priors, const uint32_t *mask, const uint8_t *pawn, int64_t B, int32_t *offsets,
                                 float *compact, void *stream) {
    if (B < 0 || !offsets || (B > 0 && (!priors || !mask || !pawn || !compact))) return aq_set_error(AQ_ERR_ARG, "aq_compact_priors");
    return compact_priors_impl(priors, mask, pawn, B, offsets, compact, AQ_WIRE_F32, reinterpret_cast<cudaStream_t>(stream));
}

// Host-buffer leaf evaluation with predict()-shaped output.  Device workspace: the dense workspace of
// aq_leaf_eval_host followed by offsets int32[B + 1] and compact [B * 136] (4 bytes per entry reserved).
static inline size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }
extern "C" int64_t aq_leaf_eval_host_compact_ws_bytes(int64_t B) {
    return aq_leaf_eval_host_ws_bytes(B) + (int64_t)align256(align16((size_t)(B + 1) * 4) + align16((size_t)B * 4) + (size_t)B * AQ_MAX_LEGAL * 4);
}
// The results of a batch form ONE block on the device: offsets int32[B+1] | value f32[B] | ragged priors, each part starting on a
// 16-byte boundary.  A caller whose host buffers have the same layout -- value_host = offsets_host + out2[0] bytes, priors_host =
// offsets_host + out2[1] bytes -- gets them with a single device -> host copy per batch instead of three.
extern "C" int aq_leaf_eval_host_compact_layout(int64_t B, int64_t *out2) {
    if (B < 0 || !out2) return aq_set_error(AQ_ERR_ARG, "aq_leaf_eval_host_compact_layout");
    out2[0] = (int64_t)align16((size_t)(B + 1) * 4);
    out2[1] = out2[0] + (int64_t)align16((size_t)B * 4);
    return 0;
}

// The call is split in two so that a caller can keep several batches in flight (one context, workspace and set of host buffers per
// batch):
//   submit: H2D of the packed states, legal mask + trunk + heads, the scan of the legal counts and the compaction, then EVERY
//           result copy of the batch -- offsets, value, optionally mask / pawn, and the ragged priors -- behind the kernels on one
//           worker stream.  The ragged array's length is only known on the device, so the priors copy is sized by a running estimate
//           the context keeps (the largest recent total plus a margin, the full capacity on the first call): no host round trip in
//           the middle of a batch;
//   wait:   one event synchronisation; in the rare case that the batch held more legal actions than the estimate, the remainder is
//           copied and waited for here.
// aq_leaf_eval_host_compact = submit + wait.
extern "C" int aq_leaf_eval_host_compact_submit(const float *params, const void *prepared, const AqState *states_host, int64_t B,
                                                void *priors_host, int64_t priors_capacity, int32_t *offsets_host, float *value_host,
                                                uint32_t *mask_host, uint8_t *pawn_host, void *dev_ws, int precision, int wire,
                                                void *host_ctx, void *stream) {
    if (B < 0 || !params || !offsets_host || !host_ctx || (B > 0 && (!states_host || !priors_host || !value_host || !dev_ws)) ||
        (wire != AQ_WIRE_F32 && wire != AQ_WIRE_F16))
        return aq_set_error(AQ_ERR_ARG, "aq_leaf_eval_host_compact");
    AqHostCtx *ctx = reinterpret_cast<AqHostCtx *>(host_ctx);
    if (ctx->pending.active) return aq_set_error(AQ_ERR_ARG, "aq_leaf_eval_host_compact_submit(a batch is already in flight on this context)");
    AqHostPending &pd = ctx->pending;
    pd = AqHostPending{};
    pd.active = true; pd.B = B; pd.priors_host = priors_host; pd.priors_capacity = priors_capacity; pd.offsets_host = offsets_host;
    pd.elem = wire == AQ_WIRE_F16 ? 2 : 4;
    pd.origin = reinterpret_cast<cudaStream_t>(stream);
    if (B == 0) return 0;
    unsigned char *p = reinterpret_cast<unsigned char *>(dev_ws);
    AqState *d_states = reinterpret_cast<AqState *>(p); p += align256((size_t)B * sizeof(AqState));
    float *d_priors = reinterpret_cast<float *>(p);     p += align256((size_t)B * kP * 4);
    p += align256((size_t)B * 4);                       // (the dense path's value array; unused here)
    uint32_t *d_mask = reinterpret_cast<uint32_t *>(p); p += align256((size_t)B * 32);
    uint8_t *d_pawn = reinterpret_cast<uint8_t *>(p);   p += align256((size_t)B * 8);
    unsigned char *d_leaf_ws = p;                       p += host_ws_region_bytes(B);
    // the result block: offsets | value | ragged priors (aq_leaf_eval_host_compact_layout)
    const size_t value_off = align16((size_t)(B + 1) * 4), priors_off = value_off + align16((size_t)B * 4);
    unsigned char *d_block = p;
    int32_t *d_offsets = reinterpret_cast<int32_t *>(d_block);
    float *d_value = reinterpret_cast<float *>(d_block + value_off);
    pd.d_compact = d_block + priors_off;

    cudaStream_t cs = ctx->s[0];
    cudaError_t e = cudaEventRecord(ctx->ready, pd.origin);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(cs, ctx->ready, 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_states, states_host, (size_t)B * sizeof(AqState), cudaMemcpyHostToDevice, cs);
    int rc = e != cudaSuccess ? aq_set_error((int)e, "aq_leaf_eval_host_compact(H2D)") : 0;
    if (!rc) rc = aq_leaf_eval(params, prepared, d_states, B, d_priors, d_value, d_mask, d_pawn, reinterpret_cast<float *>(d_leaf_ws), precision, cs);
    if (!rc) rc = compact_priors_impl(d_priors, d_mask, d_pawn, B, d_offsets, pd.d_compact, wire, cs);
    if (rc) { pd.active = false; return rc; }
    // how many ragged entries to copy without knowing the total: the context's running estimate, capped by what can exist and by
    // the caller's buffer (a too-small buffer is reported by wait(), which knows the total)
    const int64_t most = B * AQ_MAX_LEGAL;
    int64_t est = ctx->est_per_board_x1024 > 0 ? (B * ctx->est_per_board_x1024 + 1023) / 1024 + 2048 : most;
    if (est > most) est = most;
    if (est > priors_capacity) est = priors_capacity;
    pd.copied = est;
    const unsigned char *h0 = reinterpret_cast<const unsigned char *>(offsets_host);
    if (reinterpret_cast<const unsigned char *>(value_host) == h0 + value_off && reinterpret_cast<const unsigned char *>(priors_host) == h0 + priors_off) {
        // the host buffers mirror the device block: one copy for offsets, values and the estimated part of the priors
        e = cudaMemcpyAsync(offsets_host, d_block, priors_off + (size_t)est * pd.elem, cudaMemcpyDeviceToHost, cs);
    } else {
        e = cudaMemcpyAsync(offsets_host, d_offsets, (size_t)(B + 1) * 4, cudaMemcpyDeviceToHost, cs);
        if (e == cudaSuccess) e = cudaMemcpyAsync(value_host, d_value, (size_t)B * 4, cudaMemcpyDeviceToHost, cs);
        if (e == cudaSuccess && est > 0) e = cudaMemcpyAsync(priors_host, pd.d_compact, (size_t)est * pd.elem, cudaMemcpyDeviceToHost, cs);
    }
    if (e == cudaSuccess && mask_host) e = cudaMemcpyAsync(mask_host, d_mask, (size_t)B * 32, cudaMemcpyDeviceToHost, cs);
    if (e == cudaSuccess && pawn_host) e = cudaMemcpyAsync(pawn_host, d_pawn, (size_t)B * 8, cudaMemcpyDeviceToHost, cs);
    if (e == cudaSuccess) e = cudaEventRecord(ctx->chunk_done[0], cs);
    if (e != cudaSuccess) { pd.active = false; return aq_set_error((int)e, "aq_leaf_eval_host_compact(D2H)"); }
    return 0;
}

extern "C" int aq_leaf_eval_host_compact_wait(void *host_ctx) {
    if (!host_ctx) return aq_set_error(AQ_ERR_ARG, "aq_leaf_eval_host_compact_wait");
    AqHostCtx *ctx = reinterpret_cast<AqHostCtx *>(host_ctx);
    AqHostPending &pd = ctx->pending;
    if (!pd.active) return aq_set_error(AQ_ERR_ARG, "aq_leaf_eval_host_compact_wait(nothing in flight)");
    pd.active = false;
    const int64_t B = pd.B;
    if (B == 0) { pd.offsets_host[0] = 0; return 0; }
    cudaStream_t cs = ctx->s[0];
    // only this batch's own work is waited for (the worker stream), not whatever else the caller queued on `stream`
    cudaError_t e = cudaEventSynchronize(ctx->chunk_done[0]);
    if (e != cudaSuccess) return aq_set_error((int)e, "aq_leaf_eval_host_compact(sync)");
    const int64_t total = pd.offsets_host[B];
    if (total > pd.priors_capacity) return aq_set_error(AQ_ERR_ARG, "aq_leaf_eval_host_compact(priors_capacity too small)");
    if (total > pd.copied) {  // more legal actions than estimated: fetch the rest now
        e = cudaMemcpyAsync(reinterpret_cast<unsigned char *>(pd.priors_host) + (size_t)pd.copied * pd.elem,
                            pd.d_compact + (size_t)pd.copied * pd.elem, (size_t)(total - pd.copied) * pd.elem, cudaMemcpyDeviceToHost, cs);
        if (e == cudaSuccess) e = cudaStreamSynchronize(cs);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_leaf_eval_host_compact(D2H remainder)");
        ctx->short_copies++;
    }
    // running estimate of legal actions per board (x1024): jumps up to this batch's density + 3 %, decays by 1/64 per batch
    const int64_t now = (total * 1024 + B - 1) / B;
    const int64_t want = now + now / 32, decayed = ctx->est_per_board_x1024 - ctx->est_per_board_x1024 / 64;
    ctx->est_per_board_x1024 = want > decayed ? want : decayed;
    // later work on the caller's stream is ordered behind this batch
    e = cudaStreamWaitEvent(pd.origin, ctx->chunk_done[0], 0);
    if (e != cudaSuccess) return aq_set_error((int)e, "aq_leaf_eval_host_compact(join)");
    return 0;
}

extern "C" int aq_leaf_eval_host_compact(const float *params, const void *prepared /* or NULL */, const AqState *states_host, int64_t B,
                                         void *priors_host, int64_t priors_capacity, int32_t *offsets_host, float *value_host,
                                         uint32_t *mask_host, uint8_t *pawn_host, void *dev_ws, int precision, int wire, void *host_ctx,
                                         void *stream) {
    const int rc = aq_leaf_eval_host_compact_submit(params, prepared, states_host, B, priors_host, priors_capacity, offsets_host, value_host,
                                                    mask_host, pawn_host, dev_ws, precision, wire, host_ctx, stream);
    return rc ? rc : aq_leaf_eval_host_compact_wait(host_ctx);
}

// Diagnostics of a host context: [0] = batches whose ragged priors needed a second copy (estimate too small), [1] = the current
// estimate of legal actions per board x 1024.
extern "C" int aq_host_ctx_stats(void *host_ctx, int64_t *out2) {
    if (!host_ctx || !out2) return aq_set_error(AQ_ERR_ARG, "aq_host_ctx_stats");
    AqHostCtx *ctx = reinterpret_cast<AqHostCtx *>(host_ctx);
    out2[0] = ctx->short_copies;
    out2[1] = ctx->est_per_board_x1024;
    return 0;
}
