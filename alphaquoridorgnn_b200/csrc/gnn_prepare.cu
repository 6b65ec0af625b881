// aq_prepare_inference (include/aqgnn.h): the fp32 parameters -> the bf16 operand tiles of the tensor-core inference kernels
// (trunk W1 / W2 / W3 of gnn_tc2.cu, heads Wp0 / Wv0 / Wp2 of heads_tc.cu), written once per parameter update in exactly the
// shared-memory / tensor-memory layout the kernels use, so that every CTA copies instead of converting.  The counterpart of the
// reference's one-time inference preparation (BaseNetwork.py:21-32).
#include <cuda_bf16.h>
#include "gnn_fp32.cuh"
#include "tc_common.cuh"

using namespace aq;
using namespace aqtc;

namespace {
constexpr uint32_t kWKBlock = 128 * 128;  // weight tile: 128 rows x 128 B per K-block
}

// ---- aq_prepare_inference: fp32 parameters -> the bf16 operand tiles of the inference kernels ---------------------
namespace {
__global__ void prepare_inference_kernel(const float *__restrict__ params, unsigned char *__restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;  // one 16-byte output chunk per thread
    auto load8 = [&](const float *p, bool aligned, float *f) {
        if (aligned) {
            const float4 lo = __ldg(reinterpret_cast<const float4 *>(p)), hi = __ldg(reinterpret_cast<const float4 *>(p) + 1);
            f[0] = lo.x; f[1] = lo.y; f[2] = lo.z; f[3] = lo.w; f[4] = hi.x; f[5] = hi.y; f[6] = hi.z; f[7] = hi.w;
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = __ldg(p + e);
        }
    };
    float f[8];
    if (c < 4096) {  // trunk W2 / W3
        const int which = c >> 11, cc = c & 2047, n = cc >> 4, j = cc & 15;
        load8(params + (which ? kOffW3 : kOffW2) + n * kH + j * 8, true, f);
        *reinterpret_cast<uint4 *>(out + (which ? kPrepW3 : kPrepW2) + sw128_chunk(n, j, kWKBlock)) = pack8_bf16(f);
    } else if (c < 4096 + 128) {  // trunk layer-1 operand [W1 | W1 | b1_hi | b1_lo | 0 | 0]
        const int n = c - 4096;
        float w[kF];
#pragma unroll
        for (int k = 0; k < kF; ++k) w[k] = __ldg(params + kOffW1 + n * kF + k);
        const float bias = __ldg(params + kOffB1 + n);
        const float bias_hi = __bfloat162float(__float2bfloat16_rn(bias));
        uint4 c0, c1;
        c0.x = pack_bf16(w[0], w[1]); c0.y = pack_bf16(w[2], w[3]); c0.z = pack_bf16(w[4], w[5]); c0.w = pack_bf16(w[0], w[1]);
        c1.x = pack_bf16(w[2], w[3]); c1.y = pack_bf16(w[4], w[5]); c1.z = pack_bf16(bias_hi, bias - bias_hi); c1.w = 0u;
        *reinterpret_cast<uint4 *>(out + kPrepW1 + sw32_chunk(n, 0)) = c0;
        *reinterpret_cast<uint4 *>(out + kPrepW1 + sw32_chunk(n, 1)) = c1;
    } else if (c < 4096 + 128 + 2048) {  // heads B1: rows 0..63 = Wp0, 64..127 = Wv0 (Wv0 is not 16-byte aligned)
        const int cc = c - (4096 + 128), n = cc >> 4, j = cc & 15;
        if (n < kHH) load8(params + kOffWP0 + n * kH + j * 8, true, f);
        else load8(params + kOffWV0 + (n - kHH) * kH + j * 8, false, f);
        *reinterpret_cast<uint4 *>(out + kPrepHeadB1 + sw128_chunk(n, j, kWKBlock)) = pack8_bf16(f);
    } else if (c < 4096 + 128 + 2048 + 224 * 8) {  // heads B2 = Wp2 [209][64] padded to 224 rows
        const int cc = c - (4096 + 128 + 2048), n = cc >> 3, j = cc & 7;
        if (n < kP) load8(params + kOffWP2 + n * kHH + j * 8, true, f);
        else {
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = 0.f;
        }
        *reinterpret_cast<uint4 *>(out + kPrepHeadB2 + sw128_chunk(n, j, kWKBlock)) = pack8_bf16(f);
    }
}
}  // namespace

extern "C" int64_t aq_prepared_bytes(void) { return kPrepBytes; }

extern "C" int aq_prepare_inference(const float *params, void *prepared, void *stream) {
    if (!params || !prepared) return aq_set_error(AQ_ERR_ARG, "aq_prepare_inference");
    const int chunks = 4096 + 128 + 2048 + 224 * 8;
    return aq_launch("prepare_inference_kernel", prepare_inference_kernel, (chunks + 255) / 256, 256, 0, reinterpret_cast<cudaStream_t>(stream),
                     false, params, reinterpret_cast<unsigned char *>(prepared));
}
