// The optimiser step of data-parallel training as ONE kernel: fixed-order reduction of the per-CTA partial gradients,
// all-reduce of the flat 64,082-float gradient over NVLink peer memory, Adam (train_network.py:56,94) -- the counterpart of
// `loss.backward(); optimizer.step()` with torch.distributed's gradient all-reduce in between, without NCCL on the path.
//
// One process per GPU.  Every rank owns one cudaMalloc'ed communication block (two gradient slots + per-peer flag words + a step
// counter) and exports it with cudaIpcGetMemHandle; the ranks exchange the 64-byte handles (any host channel: torch.distributed's
// all_gather_object in train_network.py) and map each other's block with cudaIpcOpenMemHandle -- from then on a kernel on GPU r
// loads and stores GPU q's block directly (NVLink 5 through NVSwitch on a B200 box).
//
// dp_adam_kernel, thread of parameter pair i on rank r, step e (= the device-side step counter + 1, parity p = e & 1):
//   1. local gradient of the pair: the fixed-order slot sum of reduce_partials_kernel (deterministic), or a given flat gradient;
//   2. world > 1: PUSH the pair into the inbox every other rank keeps for rank r -- two 8-byte peer stores {value, e}: the step
//      number travels in the same 8-byte word as the value, so a word whose tag reads e carries this step's value (8-byte stores are
//      single transactions; the low-latency scheme of NCCL's LL protocol).  No fence, no block barrier, no flag round trip: measured
//      against a first version that stored into an own slot, published a flag with a system-scope release and let the peers pull
//      (15-20 us per step at two GPUs: fence + flag + pull round trip), this costs one NVLink store latency;
//      then poll the own inboxes (local memory) until the words of ranks 0 .. world-1 carry tag e and add them IN RANK ORDER (own
//      value included): every rank computes the same sum bit for bit, so the replicas never diverge.  Inboxes alternate by step
//      parity: a rank can only be one step ahead of a peer (it needs the peer's words of step e to finish step e), so a word is
//      never overwritten before it has been read;
//   3. Adam on the summed gradient (torch's lerp / addcmul / addcdiv sequence, bias corrections from the device step counter and
//      running powers of the betas in double precision);
//   4. the last CTA to finish advances the step counter.
// A rank that does not show up within kTimeoutNs (a crashed peer) makes the waiting threads give up and raise the status word, which
// aq_comm_status returns: the kernel never hangs the GPU.
// No host value changes between steps except the learning rate, so the whole training step can be captured in a CUDA graph.
#include <cmath>
#include <cstdio>
#include <cstring>
#include "gnn_fp32.cuh"

using namespace aq;

namespace {

constexpr int kMaxWorld = 8;
constexpr int kPairs = 128;                                               // parameter pairs per CTA
constexpr int kDpThreads = kPairs * 4;                                    // x 4 slot groups
constexpr int kChunkFloats = 2 * kPairs;                                  // 256 parameters per CTA
constexpr int kChunks = (kNumParams + kChunkFloats - 1) / kChunkFloats;  // 251
constexpr int kPadFloats = kChunks * kChunkFloats;
constexpr unsigned long long kTimeoutNs = 5ull * 1000 * 1000 * 1000;
static_assert(kNumParams % 2 == 0 && kOffWP0 % 2 == 0, "parameter pairs must not straddle the GCN / head boundary");

struct CommBlock {                       // layout of the exported device block
    uint2 inbox[2][kMaxWorld][kPadFloats];   // [step parity][sender][parameter] = {value bits, step tag}
    uint32_t step;                       // completed optimiser steps
    uint32_t ticket;                     // CTAs finished in the current launch
    uint32_t status;                     // != 0: a wait timed out
    uint32_t pad;
    double beta_pow[2];                  // beta1^step, beta2^step (running products: a double-precision pow() per CTA at the top of
                                         // every launch sat on the kernel's critical path)
};

struct CommPtrs {                        // passed to the kernel by value
    CommBlock *peer[kMaxWorld];
    int rank, world;
};

struct AqComm {
    CommPtrs p;
    CommBlock *local;
    cudaIpcMemHandle_t handle;
    bool opened[kMaxWorld];
};

__device__ __forceinline__ unsigned long long now_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;\n" : "=l"(t));
    return t;
}
// one 8-byte transaction each: {value, tag} never tears
__device__ __forceinline__ uint2 ld_word(const uint2 *p) {
    uint2 v;
    asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];\n" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_word(uint2 *p, uint32_t value, uint32_t tag) {
    asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};\n" ::"l"(p), "r"(value), "r"(tag) : "memory");
}

// block = 128 parameter pairs x 4 slot groups.  kFromSlots: the local gradient is the fixed-order sum of the partial slots
// (group g adds slots g, g+4, g+8, ... in that order and the four group sums are combined as (g0 + g1) + (g2 + g3): deterministic,
// four groups of independent 8-byte loads in flight per pair); otherwise it is read from grads_in.  The 128 threads of group 0
// then own one pair each for the exchange and the Adam update.
template <bool kFromSlots>
__global__ void __launch_bounds__(kDpThreads)
dp_adam_kernel(CommPtrs c, const float *grads_in, const float *partial, int gcn_slots, int head_slots, float *__restrict__ params,
               float *__restrict__ exp_avg, float *__restrict__ exp_avg_sq, float *grads_out, float lr, float beta1,
               float beta2, float eps) {
    __shared__ float2 part[4][kPairs];
    __shared__ float hyper[2];
    aq_pdl_wait();  // launched programmatically behind the backward kernels: everything read below was written before it
    const int tid = threadIdx.x, cta = blockIdx.x;
    const int tx = tid & (kPairs - 1), grp = tid / kPairs;
    CommBlock *me = c.peer[c.rank];
    const uint32_t e = *reinterpret_cast<volatile uint32_t *>(&me->step) + 1u;  // the same value in every CTA of this launch
    const int par = (int)(e & 1u);
    const double b1p = *reinterpret_cast<volatile double *>(&me->beta_pow[0]) * (double)beta1;   // beta1^e
    const double b2p = *reinterpret_cast<volatile double *>(&me->beta_pow[1]) * (double)beta2;
    if (tid == 0) {
        hyper[0] = (float)((double)lr / (1.0 - b1p));   // step_size = lr / bias_correction1
        hyper[1] = (float)sqrt(1.0 - b2p);              // bias_correction2_sqrt
    }
    const int i = cta * kChunkFloats + 2 * tx;  // this thread's parameter pair (pairs beyond kNumParams are padding)
    // the optimiser state of the pair is requested now, under the slot loads, not behind the reduction's barrier
    float2 m0 = make_float2(0.f, 0.f), v0 = m0, p0 = m0;
    if (grp == 0 && i < kNumParams) {
        m0 = *reinterpret_cast<const float2 *>(exp_avg + i);
        v0 = *reinterpret_cast<const float2 *>(exp_avg_sq + i);
        p0 = *reinterpret_cast<const float2 *>(params + i);
    }
    float2 g = make_float2(0.f, 0.f);
    if (kFromSlots) {
        if (i < kNumParams) {
            const int n = i >= kOffWP0 ? head_slots : gcn_slots;
            const float *src = partial + i;
#pragma unroll 4
            for (int k = grp; k < n; k += 4) {
                const float2 v = __ldcg(reinterpret_cast<const float2 *>(src + (int64_t)k * kNumParams));  // coherent: PDL rule
                g.x += v.x; g.y += v.y;
            }
        }
        part[grp][tx] = g;
        __syncthreads();
        if (grp == 0) {
            const float2 a = part[0][tx], b = part[1][tx], cc = part[2][tx], d = part[3][tx];
            g = make_float2((a.x + b.x) + (cc.x + d.x), (a.y + b.y) + (cc.y + d.y));
        }
    } else if (grp == 0 && i < kNumParams) {
        g = __ldcg(reinterpret_cast<const float2 *>(grads_in + i));
    }
    __syncthreads();   // hyper[]
    if (c.world > 1 && grp == 0) {
        // push this rank's pair into its inbox on every other rank
        for (int r = 0; r < c.world; ++r)
            if (r != c.rank) {
                uint2 *dst = &c.peer[r]->inbox[par][c.rank][i];
                st_word(dst, __float_as_uint(g.x), e);
                st_word(dst + 1, __float_as_uint(g.y), e);
            }
        // collect: ranks in fixed order, the own contribution in its place: bit-identical sums on every rank
        float2 a = make_float2(0.f, 0.f);
        const unsigned long long t0 = now_ns();
        bool ok = true;
        for (int r = 0; r < c.world && ok; ++r) {
            if (r == c.rank) { a.x += g.x; a.y += g.y; continue; }
            const uint2 *src = &me->inbox[par][r][i];
            uint2 w0 = ld_word(src), w1 = ld_word(src + 1);
            unsigned polls = 0;
            while (w0.y != e || w1.y != e) {
                if ((++polls & 255u) == 0u && now_ns() - t0 > kTimeoutNs) { ok = false; break; }
                w0 = ld_word(src); w1 = ld_word(src + 1);
            }
            a.x += __uint_as_float(w0.x); a.y += __uint_as_float(w1.x);
        }
        if (!ok) atomicExch(&me->status, 1u);
        g = a;
    }
    if (grp == 0 && i < kNumParams) {
        const float step_size = hyper[0], bc2_sqrt = hyper[1];
        float2 m1, v1, p1;
        m1.x = m0.x + (1.f - beta1) * (g.x - m0.x);            // exp_avg.lerp_(grad, 1 - beta1)
        m1.y = m0.y + (1.f - beta1) * (g.y - m0.y);
        v1.x = v0.x * beta2 + (1.f - beta2) * g.x * g.x;       // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
        v1.y = v0.y * beta2 + (1.f - beta2) * g.y * g.y;
        p1.x = p0.x - step_size * (m1.x / (sqrtf(v1.x) / bc2_sqrt + eps));   // (exp_avg_sq.sqrt() / bias_correction2_sqrt).add_(eps)
        p1.y = p0.y - step_size * (m1.y / (sqrtf(v1.y) / bc2_sqrt + eps));
        *reinterpret_cast<float2 *>(exp_avg + i) = m1;
        *reinterpret_cast<float2 *>(exp_avg_sq + i) = v1;
        *reinterpret_cast<float2 *>(params + i) = p1;
        if (grads_out) *reinterpret_cast<float2 *>(grads_out + i) = g;
    }
    // the last CTA of the launch advances the step counter (every CTA has read it by then: it reads it before anything else)
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(&me->ticket, 1u) == gridDim.x - 1) {
            me->ticket = 0u;
            *reinterpret_cast<volatile double *>(&me->beta_pow[0]) = b1p;
            *reinterpret_cast<volatile double *>(&me->beta_pow[1]) = b2p;
            __threadfence();
            *reinterpret_cast<volatile uint32_t *>(&me->step) = e;
        }
    }
}

}  // namespace

extern "C" int aq_comm_create(int rank, int world, void **comm, void *handle_out64) {
    if (!comm || !handle_out64 || world < 1 || world > kMaxWorld || rank < 0 || rank >= world) return aq_set_error(AQ_ERR_ARG, "aq_comm_create");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    AqComm *c = new AqComm();
    memset(&c->p, 0, sizeof c->p);
    memset(c->opened, 0, sizeof c->opened);
    c->p.rank = rank;
    c->p.world = world;
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&c->local), sizeof(CommBlock));
    if (e == cudaSuccess) e = cudaMemset(c->local, 0, sizeof(CommBlock));
    const double ones[2] = {1.0, 1.0};
    if (e == cudaSuccess) e = cudaMemcpy(&c->local->beta_pow[0], ones, sizeof ones, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess && world > 1) e = cudaIpcGetMemHandle(&c->handle, c->local);
    if (e != cudaSuccess) { if (c->local) cudaFree(c->local); delete c; return aq_set_error((int)e, "aq_comm_create"); }
    c->p.peer[rank] = c->local;
    memcpy(handle_out64, &c->handle, 64);
    *comm = c;
    return 0;
}

// handles: world x 64 bytes, entry r = what rank r's aq_comm_create returned (all ranks of ONE box)
extern "C" int aq_comm_open(void *comm, const void *handles) {
    if (!comm || !handles) return aq_set_error(AQ_ERR_ARG, "aq_comm_open");
    AqComm *c = reinterpret_cast<AqComm *>(comm);
    for (int r = 0; r < c->p.world; ++r) {
        if (r == c->p.rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, reinterpret_cast<const unsigned char *>(handles) + 64 * r, 64);
        void *ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) return aq_set_error((int)e, "aq_comm_open(cudaIpcOpenMemHandle: peer memory is not reachable)");
        c->p.peer[r] = reinterpret_cast<CommBlock *>(ptr);
        c->opened[r] = true;
    }
    return 0;
}

extern "C" int aq_comm_destroy(void *comm) {
    if (!comm) return 0;
    AqComm *c = reinterpret_cast<AqComm *>(comm);
    cudaDeviceSynchronize();
    for (int r = 0; r < kMaxWorld; ++r)
        if (c->opened[r]) cudaIpcCloseMemHandle(c->p.peer[r]);
    cudaFree(c->local);
    delete c;
    return 0;
}

// out2[0] = completed optimiser steps (the device counter), out2[1] = status (0 = ok, 1 = a peer did not arrive within the time-out).
// Synchronises the stream.
extern "C" int aq_comm_status(void *comm, int64_t *out2, void *stream) {
    if (!comm || !out2) return aq_set_error(AQ_ERR_ARG, "aq_comm_status");
    AqComm *c = reinterpret_cast<AqComm *>(comm);
    uint32_t h[4];
    cudaError_t e = cudaMemcpyAsync(h, &c->local->step, sizeof h, cudaMemcpyDeviceToHost, reinterpret_cast<cudaStream_t>(stream));
    if (e == cudaSuccess) e = cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return aq_set_error((int)e, "aq_comm_status");
    out2[0] = h[0];
    out2[1] = h[2];
    return 0;
}

// Sets the device step counter (a fresh optimiser: 0) and the running powers beta1^step, beta2^step of the bias corrections.
// Every rank must call it at the same point, with no step in flight on any rank (a host barrier before and after).
extern "C" int aq_comm_set_step(void *comm, int64_t step, float beta1, float beta2, void *stream) {
    if (!comm || step < 0) return aq_set_error(AQ_ERR_ARG, "aq_comm_set_step");
    AqComm *c = reinterpret_cast<AqComm *>(comm);
    const uint32_t v = (uint32_t)step;
    const double pw[2] = {pow((double)beta1, (double)step), pow((double)beta2, (double)step)};
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    // the inboxes are cleared too: their words carry step tags, and tags of an earlier run must not be mistaken for this one's
    cudaError_t e = cudaMemsetAsync(c->local->inbox, 0, sizeof(c->local->inbox), st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&c->local->step, &v, 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&c->local->beta_pow[0], pw, sizeof pw, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    return e == cudaSuccess ? 0 : aq_set_error((int)e, "aq_comm_set_step");
}

int aq_dp_adam_launch(void *comm, const float *grads_in, const float *partial, int gcn_slots, int head_slots, float *params, float *exp_avg,
                      float *exp_avg_sq, float *grads_out, float lr, float beta1, float beta2, float eps, bool pdl, cudaStream_t st) {
    AqComm *c = reinterpret_cast<AqComm *>(comm);
    if (partial)
        return aq_launch("dp_adam_kernel", dp_adam_kernel<true>, kChunks, kDpThreads, 0, st, pdl, c->p, grads_in, partial, gcn_slots, head_slots,
                         params, exp_avg, exp_avg_sq, grads_out, lr, beta1, beta2, eps);
    return aq_launch("dp_adam_kernel", dp_adam_kernel<false>, kChunks, kDpThreads, 0, st, pdl, c->p, grads_in, partial, gcn_slots, head_slots,
                     params, exp_avg, exp_avg_sq, grads_out, lr, beta1, beta2, eps);
}

// All-reduce (sum over the ranks of `comm`) of a flat gradient + Adam step, one kernel.  grads: this rank's gradient (n = 64,082
// floats, flat parameter order); on return of the kernel it holds the SUM over the ranks (what torch.distributed.all_reduce leaves).
// The step number of the bias corrections is the communicator's device counter + 1 (aq_comm_set_step / aq_comm_status).
extern "C" int aq_dp_adam_step(void *comm, float *params, float *grads, float *exp_avg, float *exp_avg_sq, float lr, float beta1, float beta2,
                               float eps, void *stream) {
    if (!comm || !params || !grads || !exp_avg || !exp_avg_sq) return aq_set_error(AQ_ERR_ARG, "aq_dp_adam_step");
    return aq_dp_adam_launch(comm, grads, nullptr, 0, 0, params, exp_avg, exp_avg_sq, grads, lr, beta1, beta2, eps, false,
                             reinterpret_cast<cudaStream_t>(stream));
}
