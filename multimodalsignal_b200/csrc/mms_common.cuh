// Shared device/host helpers for libmms_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/mms_b200.h"

namespace mms {

// ---- error plumbing ------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define MMS_CUDA(call)                                                              \
    do {                                                                            \
        cudaError_t _e = (call);                                                    \
        if (_e != cudaSuccess) return ::mms::cuda_fail(_e, #call, __FILE__, __LINE__); \
    } while (0)

// Launch bookkeeping: every kernel launch is preceded by MMS_PROF_BEGIN(stream) and followed by
// MMS_LAUNCH_CHECK(name).  Both are a counter increment unless mms_profile_enable(1) was called, in
// which case the launch is bracketed by CUDA events on its stream (bench.py's live kernel times).
void prof_begin(cudaStream_t st);
void prof_end(const char* name);

#define MMS_PROF_BEGIN(st) ::mms::prof_begin(st)

#define MMS_LAUNCH_CHECK(name)                                                      \
    do {                                                                            \
        cudaError_t _e = cudaPeekAtLastError();                                     \
        if (_e != cudaSuccess) return ::mms::cuda_fail(_e, name, __FILE__, __LINE__);  \
        ::mms::prof_end(name);                                                      \
    } while (0)

#define MMS_REQUIRE(cond, ...)                                                      \
    do {                                                                            \
        if (!(cond)) { ::mms::set_error(__VA_ARGS__); return MMS_E_INVALID; }       \
    } while (0)

// Integer run-time switches (A/B measurements, opt-in kernels): the value set by mms_set_option(name, v) wins, else the
// environment variable MMS_<name> read once, else `dflt`.
int option_get(const char* name, int dflt);

// One weight-gradient (TN) product, the argument list of launch_tc_gemm_tn / mms_gemm_tn_acc as a record, so that the
// products of a GRU layer can be handed to the batched tensor-core kernel in one call.
struct TnCall {
    const float* A; int64_t lda; int a_split, a_skip;
    const float* Bm; int64_t ldb; int shift, seq;
    float* C; int64_t ldc; float* bias_grad;
    int M, N1, N2;
};

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a PER-DEVICE property of a kernel: the opt-in guards at the launch
// sites remember it per device (several devices in one process: mms_init(dev), per-device side streams), not per process.
struct PerDeviceOnce {
    bool done[64] = {};
    bool need() {
        int d = 0;
        cudaGetDevice(&d);
        d &= 63;
        if (done[d]) return false;
        done[d] = true;
        return true;
    }
};

static inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }
static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- shapes of the reference CNN stack (models.py:46-53) ------------------------------
static inline int conv_out_len(int l_in, int k, int s, int p) { return (l_in + 2 * p - k) / s + 1; }
static inline int pool_out_len(int l_in) { return (l_in + 2 - 3) / 2 + 1; }

constexpr int CONV1_CO = 16, CONV1_K = 7, CONV1_S = 2, CONV1_P = 3;
constexpr int CONV2_CI = 16, CONV2_K = 5, CONV2_S = 2, CONV2_P = 2;
constexpr int HEAD_HID = 64;
constexpr float BN_EPS = 1e-5f;
constexpr float BN_MOMENTUM = 0.1f;

// BatchNorm backward folded into the consumers of a conv layer's output gradient (conv1d_dgrad / conv1d_wgrad): when
// y != nullptr the `dy` those kernels are given is the UN-normalised gradient dyn = d(relu/pool) and they form
//     dy = a * (dyn - mean(dyn) - xhat * mean(dyn * xhat)),   a = gamma / sqrt(var + eps),  xhat = (y - mean) / sqrt(var + eps)
// themselves while staging their tile (red = the two float64 reductions of pool_relu_bwd; eval mode: dy = a * dyn), which
// removes the separate BN-apply pass (one launch and one read + write of the whole gradient) from the critical path.
// dgamma / dbeta (optional) are added once, by the weight-gradient kernel.
struct BnBwd {
    const float* y;
    const double* stats;
    const float* gamma;
    const float* beta;
    const float* rm;
    const float* rv;
    const double* red;
    float* dgamma;
    float* dbeta;
    int Bstat;
    int training;
    float grad_scale;
};

// Flat ranges of the Adam update (mms_adam_ranges_step), passed by value: range k is [off[k], off[k] + cnt[k]) with step
// counter steps[slot[k]].
struct AdamRanges {
    int n;
    int64_t off[MMS_MAX_ADAM_RANGES], cnt[MMS_MAX_ADAM_RANGES];
    int32_t slot[MMS_MAX_ADAM_RANGES];
};
// Reads a HOST (offset, count, slot) table; every range must lie inside [0, total) and be disjoint from the others.
int adam_ranges_from_host(const int64_t* table, int n, int64_t total, AdamRanges* r);

// ---- programmatic dependent launch (build variant, -DMMS_PDL; default build: every macro below is a no-op) ---------
// 25 dependent launches make up the critical path of a step, and each edge costs the drain of the producer plus the launch,
// CTA scheduling and prologue of the consumer.  With MMS_PDL the kernels of the main chain are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization: MMS_PDL_TRIGGER() (griddepcontrol.launch_dependents) at the top of a
// kernel lets the NEXT kernel of the stream start while this one runs, and that kernel executes MMS_PDL_WAIT()
// (griddepcontrol.wait: every prerequisite grid complete and its memory visible) before it touches anything an earlier
// kernel of the step wrote or still reads -- after its weight / invariant prologue where that prologue only reads
// parameters (constant within a step; the first kernel of a step is not launched this way).  Rule: a kernel may be passed to
// MMS_LAUNCH only if it executes MMS_PDL_WAIT() on every path before its first such access.  The first kernel of the
// forward and of the backward pass follows a memset node (full dependency) and chan_gate is a plain launch, so every kernel
// of a step starts after the previous step's Adam has completed: reading parameters ahead of the wait is safe.
// Build: MMS_NVCC_EXTRA="-DMMS_PDL" python -m multimodalsignal_b200.build --force   (parity-green on a B200 but slower than the default build in round 2: not the default)
#ifdef MMS_PDL
#define MMS_PDL_TRIGGER() asm volatile("griddepcontrol.launch_dependents;" ::: "memory")
#define MMS_PDL_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
#else
#define MMS_PDL_TRIGGER() ((void)0)
#define MMS_PDL_WAIT() ((void)0)
#endif
#define MMS_PDL_PROLOGUE() do { MMS_PDL_TRIGGER(); MMS_PDL_WAIT(); } while (0)

// ---- device helpers -----------------------------------------------------------------
#ifdef __CUDACC__

#ifdef MMS_PDL
template <typename... KArgs, typename... Args>
static inline void pdl_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);      // errors surface in MMS_LAUNCH_CHECK (cudaPeekAtLastError)
}
#define MMS_LAUNCH(kern, grid, block, smem, st, ...) ::mms::pdl_launch(kern, grid, block, smem, st, __VA_ARGS__)
#else
#define MMS_LAUNCH(kern, grid, block, smem, st, ...) kern<<<grid, block, smem, st>>>(__VA_ARGS__)
#endif

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Counter-based dropout stream: murmur3 finaliser over (seed, offset, element index).
// Not bit-compatible with torch's Philox stream (nothing outside torch can be).  oracle/dropout_stream.py
// ports it to the host and states the element ids of every dropout site; tests/test_gpu_dropout.py pins
// the port to these kernels bit for bit and checks training steps with dropout against the float64
// oracle, with the masks the kernels drew rebuilt from (seed, offset, id).
__device__ __forceinline__ uint32_t fmix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    return h;
}
struct DropRng {
    uint32_t k0, k1;
    float p, scale;
    __device__ __forceinline__ void init(uint64_t seed, uint64_t offset, float p_) {
        k0 = fmix32((uint32_t)seed ^ 0x9e3779b9u) ^ fmix32((uint32_t)(offset) + 0x7f4a7c15u);
        k1 = fmix32((uint32_t)(seed >> 32) ^ 0x85ebca6bu) + fmix32((uint32_t)(offset >> 32) ^ 0xc2b2ae35u);
        p = p_;
        scale = p_ < 1.f ? 1.f / (1.f - p_) : 0.f;
    }
    // multiplier applied to element `idx`: 0 (dropped) or 1/(1-p)
    __device__ __forceinline__ float mult(uint64_t idx) const {
        uint32_t h = fmix32((uint32_t)idx ^ k0);
        h = fmix32(h + k1 + (uint32_t)(idx >> 32) * 0x27d4eb2fu);
        float u = (float)(h >> 8) * (1.0f / 16777216.0f);
        return u >= p ? scale : 0.f;
    }
};

__device__ __forceinline__ uint64_t resolve_offset(uint64_t host_off, const int64_t* dev_off) {
    return dev_off ? (uint64_t)(*dev_off) : host_off;
}

__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }

// torch.optim.Adam single-tensor rule (coupled L2 weight decay), shared by every Adam kernel of the library:
//   g += wd*p; m = b1*m + (1-b1)*g; v = b2*v + (1-b2)*g*g;
//   p -= (lr / (1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps),   t = steps_done + 1
struct AdamCoef {
    float step_size, bc2_sqrt;
};
__device__ __forceinline__ AdamCoef adam_coef(int64_t steps_done, float lr, float beta1, float beta2) {
    const double t = (double)(steps_done + 1);
    const float bc1 = (float)(1.0 - pow((double)beta1, t));
    const float bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, t));
    return {lr / bc1, bc2_sqrt};
}
// element i, the gradient read from g[i]
__device__ __forceinline__ void adam_update(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                            float* __restrict__ v, int64_t i, const AdamCoef c, float beta1, float beta2, float eps,
                                            float wd) {
    const float pi = p[i];
    const float gi = g[i] + wd * pi;
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / c.bc2_sqrt + eps;
    p[i] = pi - c.step_size * (mi / denom);
}
// the same for one element of registers whose gradient has already been summed (the peer kernels)
__device__ __forceinline__ float adam_update(float pi, float gsum, float& mi, float& vi, const AdamCoef c, float beta1, float beta2,
                                             float eps, float wd) {
    const float gi = gsum + wd * pi;
    mi = beta1 * mi + (1.f - beta1) * gi;
    vi = beta2 * vi + (1.f - beta2) * gi * gi;
    return pi - c.step_size * (mi / (sqrtf(vi) / c.bc2_sqrt + eps));
}

// ---- gradient-norm clipping (torch.nn.utils.clip_grad_norm_, norm_type 2; grad_clip.cu, peer.cu) ----------------------
// The norm kernels stride over the virtual index space of an AdamRanges table (the ranges laid end to end, as in
// adam_ranges_kernel), so the element -> thread map, and with it the float64 sum, depends only on the concatenated ranges and
// the grid size, which grad_norm_blocks fixes from the element count: the norm is bit-reproducible, and the same whether the
// trainable elements are listed per segment or per tensor.  Each CTA writes one float64 partial; the last CTA to arrive adds
// them in CTA order.
constexpr int GRAD_NORM_MAX_CTAS = 128;
struct ClipScratch {                       // mms_cnngru_desc.clip_scratch, MMS_GRAD_CLIP_SCRATCH_BYTES, zero-initialised
    float norm;                            // this step's total norm before clipping (fp32)
    float coef;                            // clamp(max_norm / (norm + 1e-6), max = 1), what the clipped Adam multiplies by
    uint32_t arrived;                      // CTAs done (the last one resets it)
    uint32_t pad;
    double partial[GRAD_NORM_MAX_CTAS];
};
static_assert(sizeof(ClipScratch) == MMS_GRAD_CLIP_SCRATCH_BYTES, "ClipScratch layout");

static inline int grad_norm_blocks(int64_t n) {
    const int64_t b = (n + 1023) / 1024;
    return (int)(b < 1 ? 1 : (b > GRAD_NORM_MAX_CTAS ? GRAD_NORM_MAX_CTAS : b));
}

// torch's coefficient bit for bit: max_norm / t is Tensor.__rtruediv__ = t.reciprocal() * max_norm, and torch.clamp(max=1)
// keeps a NaN (fminf would not)
__device__ __forceinline__ float clip_coef(float norm, float max_norm) {
    const float c = __fmul_rn(__frcp_rn(__fadd_rn(norm, 1e-6f)), max_norm);
    return c > 1.f ? 1.f : c;
}

// Block-reduces `sumsq` (every thread of the CTA calls it), publishes the CTA's partial and, in the last CTA to arrive,
// writes the norm and the coefficient and adds this step to the record: [0] sum of the finite norms, [1] their maximum,
// [2] steps with coef < 1, [3] steps with a non-finite norm, [4] steps.  No CTA waits for another.  True in the one thread
// that finished the step.
__device__ __forceinline__ bool grad_norm_finish(double sumsq, ClipScratch* cs, const float* __restrict__ max_norm_dev,
                                                 double* record) {
    __shared__ double s_w[32];
    sumsq = warp_sum(sumsq);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = sumsq;
    __syncthreads();
    if (threadIdx.x != 0) return false;
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += s_w[w];
    cs->partial[blockIdx.x] = s;
    __threadfence();
    if (atomicAdd(&cs->arrived, 1u) != gridDim.x - 1) return false;
    __threadfence();
    const volatile double* part = cs->partial;
    double total = 0.0;
    for (int b = 0; b < (int)gridDim.x; ++b) total += part[b];
    const float norm = (float)sqrt(total);
    const float coef = clip_coef(norm, *max_norm_dev);
    cs->norm = norm;
    cs->coef = coef;
    cs->arrived = 0u;
    if (record) {
        if (isfinite(norm)) {
            record[0] += (double)norm;
            record[1] = fmax(record[1], (double)norm);
        } else {
            record[3] += 1.0;
        }
        if (coef < 1.f) record[2] += 1.0;
        record[4] += 1.0;
    }
    return true;
}

// adam_update with the gradient scaled first: torch clips p.grad in place, and Adam adds wd * p to the ROUNDED product
// (__fmul_rn is never contracted into the FMA that follows).  coef == 1 gives adam_update's result bit for bit.
__device__ __forceinline__ void adam_update_clipped(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                    float* __restrict__ v, int64_t i, float coef, const AdamCoef c, float beta1,
                                                    float beta2, float eps, float wd) {
    const float pi = p[i];
    const float gi = __fmul_rn(g[i], coef) + wd * pi;
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / c.bc2_sqrt + eps;
    p[i] = pi - c.step_size * (mi / denom);
}

#endif  // __CUDACC__

}  // namespace mms
