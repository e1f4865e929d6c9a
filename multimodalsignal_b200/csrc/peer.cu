// Intra-fold data parallelism without a communication library on the data path (SURVEY §8e, BASELINE configs[4]):
// the two exchange steps of a data-parallel training step -- the SyncBN statistics (<= 1 KB, four times per step) and
// the flat gradient buffer (0.5 MB, once) -- are done by kernels that read the peers' buffers directly over NVLink
// (the buffers live in symmetric memory mapped into every rank's address space) and synchronise through flags in the
// peers' signal pads.  The gradient all-reduce is FUSED with Adam (reference trainer.py:148-149): every rank sums the
// world's gradient buffers on the fly, in rank order (bit-identical parameters on all ranks), and applies the update;
// the reduced gradient is never written anywhere.
//
// Cross-GPU barrier ("everybody has passed point X of epoch e"): rank r stores e into word [base + r] of EVERY peer's
// signal pad (st.release.sys after a system fence) and then spins until all `world` words of its OWN pad are >= e
// (ld.acquire.sys).  Epochs only grow, so the words never need resetting; `epoch_dev` (local) holds the last epoch used.
// Each call uses two barriers: "my data is ready" before the peers are read, and "I have finished reading" before the
// kernel ends, so that whatever runs next on any rank may overwrite its buffer.
//
// Failure behaviour: every wait is BOUNDED (%globaltimer deadline, MMS_PEER_TIMEOUT_MS, default 2000 ms).  A rank that has
// died, diverged in step count or raised on the host between two phases therefore cannot hang the other GPUs inside a
// kernel that nothing short of a device reset could cancel: the waiting threads give up, count the event in a device
// counter and the kernel finishes (with a meaningless sum); mms_peer_status() reads and clears the counter, and the Python
// side checks it wherever it reads a loss back (parallel.DataParallelTrainStep.global_loss) and raises.
// No kernel here depends on its own CTAs being co-resident: every CTA of the fused Adam kernel polls the rank's own signal
// pad itself (CTA 0, which the hardware dispatches first, is the only one that signals the peers), and the closing barrier
// is run by whichever CTA finishes last.
#include "mms_common.cuh"

namespace mms {

constexpr int PEER_MAX_WORLD = 16;

struct PeerPtrs {
    const void* buf[PEER_MAX_WORLD];       // the peers' copies of the buffer (buf[rank] is the local one)
    uint32_t* sig[PEER_MAX_WORLD];         // the peers' signal pads
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.global.release.sys.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.global.acquire.sys.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_relaxed_sys_f4(const float* p) {
    float4 v;
    asm volatile("ld.global.relaxed.sys.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ld_relaxed_sys_f(const float* p) {
    float v;
    asm volatile("ld.global.relaxed.sys.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_relaxed_sys_d(const double* p) {
    double v;
    asm volatile("ld.global.relaxed.sys.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

__device__ unsigned int g_peer_timeouts;      // waits that ran into their deadline since the last mms_peer_status()

__device__ __forceinline__ uint64_t globaltimer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// spin until *word >= e (epochs wrap: signed difference) or `timeout_ns` has passed; false + one count on a timeout
__device__ __forceinline__ bool spin_until(const uint32_t* word, uint32_t e, uint64_t timeout_ns) {
    if ((int32_t)(ld_acquire_sys(word) - e) >= 0) return true;
    const uint64_t t0 = globaltimer_ns();
    for (;;) {
#pragma unroll 1
        for (int i = 0; i < 64; ++i)
            if ((int32_t)(ld_acquire_sys(word) - e) >= 0) return true;
        if (globaltimer_ns() - t0 > timeout_ns) {
            atomicAdd(&g_peer_timeouts, 1u);
            return false;
        }
    }
}

// "I have passed this point of epoch e": threads 0 .. world-1 of ONE CTA store e into every peer's pad
__device__ __forceinline__ void peer_signal(const PeerPtrs& pp, int world, int rank, int base, uint32_t e, int tid) {
    if (tid < world) {
        __threadfence_system();
        st_release_sys(pp.sig[tid] + base + rank, e);
    }
}
// "every rank has passed it": threads 0 .. world-1 wait on the words of the rank's OWN pad; the caller synchronises the CTA
__device__ __forceinline__ void peer_wait(const PeerPtrs& pp, int world, int rank, int base, uint32_t e, int tid, uint64_t timeout_ns) {
    if (tid < world) spin_until(pp.sig[rank] + base + tid, e, timeout_ns);
}
__device__ __forceinline__ void peer_barrier(const PeerPtrs& pp, int world, int rank, int base, uint32_t e, int tid, uint64_t timeout_ns) {
    peer_signal(pp, world, rank, base, e, tid);
    peer_wait(pp, world, rank, base, e, tid, timeout_ns);
}

// v[i] = sum over the ranks (rank order) of buf[p][i], i < count <= blockDim.x, written back IN PLACE to the local buffer
// after every peer has finished reading it.  One CTA.
__global__ void __launch_bounds__(256) peer_allreduce_f64_kernel(const PeerPtrs pp, int world, int rank, int base, int count,
                                                                 uint32_t* epoch_dev, uint64_t timeout_ns) {
    const int tid = threadIdx.x;
    const uint32_t e = *epoch_dev + 1;
    __syncthreads();                               // everybody has read the epoch before thread 0 advances it
    peer_barrier(pp, world, rank, base, e, tid, timeout_ns);   // the peers' values are in place
    __syncthreads();
    double s = 0.0;
    if (tid < count)
        for (int p = 0; p < world; ++p) s += ld_relaxed_sys_d(reinterpret_cast<const double*>(pp.buf[p]) + tid);
    __syncthreads();
    peer_barrier(pp, world, rank, base + world, e, tid, timeout_ns);    // everybody has read everybody
    __syncthreads();
    if (tid < count) const_cast<double*>(reinterpret_cast<const double*>(pp.buf[rank]))[tid] = s;
    if (tid == 0) *epoch_dev = e;
}

// Fused gradient all-reduce + Adam (adam_update, the rule of adam_flat_kernel in head_opt.cu).  CTA 0 tells the peers that this
// rank's gradient is complete; EVERY CTA waits for the peers' signals on the rank's own pad (no CTA waits for another CTA of
// the same launch, so nothing depends on co-residency); the last CTA to finish runs the closing barrier.
// RANGES: only the elements of `r` are summed and updated, range k with its own step count steps[r.slot[k]] (see
// adam_ranges_kernel); otherwise the whole buffer with *step_dev.
// CLIP: the summed gradient is scaled by *coef_dev (mms_peer_grad_norm) before the update, rounded before + wd * p.
template <bool RANGES, bool CLIP = false>
__device__ __forceinline__ void peer_adam_body(float* __restrict__ p, const PeerPtrs& pp, float* __restrict__ m, float* __restrict__ v,
                                               int64_t n, const AdamRanges* r, int64_t* steps, const float* __restrict__ lr_dev,
                                               float beta1, float beta2, float eps, float wd, int64_t* step_dev, int world, int rank,
                                               int base, uint32_t* epoch_dev, uint32_t* done_dev, uint64_t timeout_ns,
                                               const float* __restrict__ coef_dev = nullptr) {
    const int tid = threadIdx.x;
    const uint32_t e = *epoch_dev + 1;
    const float lr = *lr_dev;
    const float coef = CLIP ? *coef_dev : 1.f;
    __shared__ AdamCoef s_c[RANGES ? MMS_MAX_ADAM_RANGES : 1];
    if (RANGES)
        for (int k = tid; k < r->n; k += blockDim.x) s_c[k] = adam_coef(steps[r->slot[k]], lr, beta1, beta2);
    const AdamCoef c = RANGES ? AdamCoef{0.f, 0.f} : adam_coef(*step_dev, lr, beta1, beta2);
    if (blockIdx.x == 0) peer_signal(pp, world, rank, base, e, tid);      // this rank's gradient buffer is complete (stream order)
    peer_wait(pp, world, rank, base, e, tid, timeout_ns);                   // ... and so is every peer's
    __syncthreads();
    if (RANGES) {
        const int64_t stride = (int64_t)gridDim.x * blockDim.x, gt = (int64_t)blockIdx.x * blockDim.x + tid;
        int64_t vbase = 0;
        for (int k = 0; k < r->n; ++k) {
            const AdamCoef ck = s_c[k];
            int64_t j = (gt - vbase) % stride;
            if (j < 0) j += stride;
            for (; j < r->cnt[k]; j += stride) {
                const int64_t i = r->off[k] + j;
                float g = 0.f;
                for (int q = 0; q < world; ++q) g += ld_relaxed_sys_f(reinterpret_cast<const float*>(pp.buf[q]) + i);
                if (CLIP) g = __fmul_rn(g, coef);
                float mi = m[i], vi = v[i];
                p[i] = adam_update(p[i], g, mi, vi, ck, beta1, beta2, eps, wd);
                m[i] = mi;
                v[i] = vi;
            }
            vbase += r->cnt[k];
        }
    } else {
        const int64_t n4 = n >> 2;
        for (int64_t i4 = (int64_t)blockIdx.x * blockDim.x + tid; i4 < n4; i4 += (int64_t)gridDim.x * blockDim.x) {
            float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int q = 0; q < world; ++q) {
                const float4 x = ld_relaxed_sys_f4(reinterpret_cast<const float*>(pp.buf[q]) + 4 * i4);
                g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
            }
            if (CLIP) { g.x = __fmul_rn(g.x, coef); g.y = __fmul_rn(g.y, coef); g.z = __fmul_rn(g.z, coef); g.w = __fmul_rn(g.w, coef); }
            float4 pv = reinterpret_cast<float4*>(p)[i4], mv = reinterpret_cast<float4*>(m)[i4], vv = reinterpret_cast<float4*>(v)[i4];
            float* gp = &g.x; float* pq = &pv.x; float* mq = &mv.x; float* vq = &vv.x;
#pragma unroll
            for (int j = 0; j < 4; ++j) pq[j] = adam_update(pq[j], gp[j], mq[j], vq[j], c, beta1, beta2, eps, wd);
            reinterpret_cast<float4*>(p)[i4] = pv;
            reinterpret_cast<float4*>(m)[i4] = mv;
            reinterpret_cast<float4*>(v)[i4] = vv;
        }
        if (blockIdx.x == 0) {                                 // tail (n is a multiple of 4 for every supported layout; kept for safety)
            for (int64_t i = (n4 << 2) + tid; i < n; i += blockDim.x) {
                float g = 0.f;
                for (int q = 0; q < world; ++q) g += ld_relaxed_sys_f(reinterpret_cast<const float*>(pp.buf[q]) + i);
                if (CLIP) g = __fmul_rn(g, coef);
                p[i] = adam_update(p[i], g, m[i], v[i], c, beta1, beta2, eps, wd);
            }
        }
    }
    __syncthreads();
    // the last CTA to finish tells the peers that this rank no longer reads their gradients, waits for the same from
    // them (so that the next step may zero / overwrite the local buffer) and advances the counters
    __shared__ int s_last;
    if (tid == 0) {
        __threadfence();
        s_last = atomicAdd(done_dev, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (s_last) {
        peer_barrier(pp, world, rank, base + world, e, tid, timeout_ns);
        __syncthreads();
        if (tid == 0) {
            *done_dev = 0u;
            *epoch_dev = e;
            *step_dev += 1;
            if (RANGES)
                for (int k = 0; k < r->n; ++k) steps[r->slot[k]] += 1;
        }
    }
}

__global__ void __launch_bounds__(256) peer_allreduce_adam_kernel(float* __restrict__ p, const PeerPtrs pp, float* __restrict__ m,
                                                                  float* __restrict__ v, int64_t n, const float* __restrict__ lr_dev,
                                                                  float beta1, float beta2, float eps, float wd, int64_t* step_dev,
                                                                  int world, int rank, int base, uint32_t* epoch_dev,
                                                                  uint32_t* done_dev, uint64_t timeout_ns) {
    peer_adam_body<false>(p, pp, m, v, n, nullptr, nullptr, lr_dev, beta1, beta2, eps, wd, step_dev, world, rank, base, epoch_dev,
                          done_dev, timeout_ns);
}

__global__ void __launch_bounds__(256) peer_allreduce_adam_ranges_kernel(float* __restrict__ p, const PeerPtrs pp, float* __restrict__ m,
                                                                         float* __restrict__ v, const __grid_constant__ AdamRanges r,
                                                                         int64_t* steps, const float* __restrict__ lr_dev, float beta1,
                                                                         float beta2, float eps, float wd, int64_t* step_dev, int world,
                                                                         int rank, int base, uint32_t* epoch_dev, uint32_t* done_dev,
                                                                         uint64_t timeout_ns) {
    peer_adam_body<true>(p, pp, m, v, 0, &r, steps, lr_dev, beta1, beta2, eps, wd, step_dev, world, rank, base, epoch_dev, done_dev,
                         timeout_ns);
}

__global__ void __launch_bounds__(256) peer_allreduce_adam_clip_kernel(float* __restrict__ p, const PeerPtrs pp, float* __restrict__ m,
                                                                       float* __restrict__ v, int64_t n, const float* __restrict__ lr_dev,
                                                                       float beta1, float beta2, float eps, float wd, int64_t* step_dev,
                                                                       int world, int rank, int base, uint32_t* epoch_dev,
                                                                       uint32_t* done_dev, uint64_t timeout_ns,
                                                                       const float* __restrict__ coef_dev) {
    peer_adam_body<false, true>(p, pp, m, v, n, nullptr, nullptr, lr_dev, beta1, beta2, eps, wd, step_dev, world, rank, base, epoch_dev,
                                done_dev, timeout_ns, coef_dev);
}

__global__ void __launch_bounds__(256) peer_allreduce_adam_ranges_clip_kernel(float* __restrict__ p, const PeerPtrs pp,
                                                                              float* __restrict__ m, float* __restrict__ v,
                                                                              const __grid_constant__ AdamRanges r, int64_t* steps,
                                                                              const float* __restrict__ lr_dev, float beta1, float beta2,
                                                                              float eps, float wd, int64_t* step_dev, int world, int rank,
                                                                              int base, uint32_t* epoch_dev, uint32_t* done_dev,
                                                                              uint64_t timeout_ns, const float* __restrict__ coef_dev) {
    peer_adam_body<true, true>(p, pp, m, v, 0, &r, steps, lr_dev, beta1, beta2, eps, wd, step_dev, world, rank, base, epoch_dev,
                               done_dev, timeout_ns, coef_dev);
}

// The norm of the world's summed gradient over the virtual index space of `r` (grad_norm_kernel, grad_clip.cu), every element
// summed over the ranks in rank order with the fp32 additions of peer_adam_body, so that every rank forms the same norm and
// coefficient.  CTA 0 signals "this rank's gradient is complete" on words [base, base + world) with its own epoch; every CTA
// waits for the peers on the rank's own pad.  No closing barrier: the clipped Adam kernel that follows signals again and ends
// with the barrier after which the gradient buffers may be overwritten.
__global__ void __launch_bounds__(256) peer_grad_norm_kernel(const PeerPtrs pp, int world, int rank, int base,
                                                             const __grid_constant__ AdamRanges r, const float* __restrict__ max_norm_dev,
                                                             double* record, ClipScratch* cs, uint32_t* epoch_dev, uint64_t timeout_ns) {
    const int tid = threadIdx.x;
    const uint32_t e = *epoch_dev + 1;
    if (blockIdx.x == 0) peer_signal(pp, world, rank, base, e, tid);
    peer_wait(pp, world, rank, base, e, tid, timeout_ns);
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, gt = (int64_t)blockIdx.x * blockDim.x + tid;
    double s = 0.0;
    int64_t vbase = 0;
    for (int k = 0; k < r.n; ++k) {
        int64_t j = (gt - vbase) % stride;
        if (j < 0) j += stride;
        for (; j < r.cnt[k]; j += stride) {
            const int64_t i = r.off[k] + j;
            float g = 0.f;
            for (int q = 0; q < world; ++q) g += ld_relaxed_sys_f(reinterpret_cast<const float*>(pp.buf[q]) + i);
            const double x = (double)g;
            s += x * x;
        }
        vbase += r.cnt[k];
    }
    // the last CTA to arrive advances the epoch: every CTA read it before it arrived
    if (grad_norm_finish(s, cs, max_norm_dev, record)) *epoch_dev = e;
}

static int fill_peer(PeerPtrs* pp, const void* const* bufs_host, void* const* signals_host, int world) {
    MMS_REQUIRE(world >= 1 && world <= PEER_MAX_WORLD, "peer: world size %d outside [1,%d]", world, PEER_MAX_WORLD);
    for (int i = 0; i < PEER_MAX_WORLD; ++i) {
        pp->buf[i] = i < world ? bufs_host[i] : nullptr;
        pp->sig[i] = i < world ? reinterpret_cast<uint32_t*>(signals_host[i]) : nullptr;
        MMS_REQUIRE(i >= world || (pp->buf[i] && pp->sig[i]), "peer: null peer pointer");
    }
    return MMS_OK;
}

static uint64_t peer_timeout_ns() {
    int ms = option_get("PEER_TIMEOUT_MS", 2000);
    if (ms < 1) ms = 1;
    return (uint64_t)ms * 1000000ull;
}

}  // namespace mms

using namespace mms;

// Number of peer waits that ran into their deadline on the current device since the last call (read and cleared; synchronises).
extern "C" int mms_peer_status(uint32_t* timeouts_host) {
    MMS_REQUIRE(timeouts_host, "peer_status: null pointer");
    unsigned int v = 0, zero = 0;
    MMS_CUDA(cudaMemcpyFromSymbol(&v, g_peer_timeouts, sizeof(v)));
    if (v) MMS_CUDA(cudaMemcpyToSymbol(g_peer_timeouts, &zero, sizeof(zero)));
    *timeouts_host = v;
    return MMS_OK;
}

extern "C" int mms_peer_allreduce_f64(const void* const* bufs_host, void* const* signals_host, int32_t world, int32_t rank,
                                      int32_t signal_base, int32_t count, uint32_t* epoch_dev, mms_stream_t stream) {
    MMS_REQUIRE(bufs_host && signals_host && epoch_dev && rank >= 0 && rank < world && count >= 1 && count <= 256 && signal_base >= 0,
                "peer_allreduce_f64: bad arguments");
    PeerPtrs pp;
    int rc = fill_peer(&pp, bufs_host, signals_host, world);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    peer_allreduce_f64_kernel<<<1, 256, 0, st>>>(pp, world, rank, signal_base, count, epoch_dev, peer_timeout_ns());
    MMS_LAUNCH_CHECK("peer_allreduce_f64_kernel");
    return MMS_OK;
}

extern "C" int mms_peer_allreduce_adam(float* params, const void* const* grads_host, void* const* signals_host, int32_t world,
                                       int32_t rank, int32_t signal_base, float* exp_avg, float* exp_avg_sq, int64_t n,
                                       const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                                       int64_t* step_dev, uint32_t* epoch_dev, uint32_t* scratch2_dev, mms_stream_t stream) {
    MMS_REQUIRE(params && grads_host && signals_host && exp_avg && exp_avg_sq && lr_dev && step_dev && epoch_dev && scratch2_dev &&
                    rank >= 0 && rank < world && n > 0 && signal_base >= 0,
                "peer_allreduce_adam: bad arguments");
    MMS_REQUIRE(((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(exp_avg) | reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0,
                "peer_allreduce_adam: buffers must be 16-byte aligned");
    PeerPtrs pp;
    int rc = fill_peer(&pp, grads_host, signals_host, world);
    if (rc) return rc;
    for (int i = 0; i < world; ++i) MMS_REQUIRE((reinterpret_cast<uintptr_t>(pp.buf[i]) & 15) == 0, "peer_allreduce_adam: gradient buffers must be 16-byte aligned");
    int blocks = (int)((n / 4 + 255) / 256);
    if (blocks > 64) blocks = 64;
    if (blocks < 1) blocks = 1;
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    peer_allreduce_adam_kernel<<<blocks, 256, 0, st>>>(params, pp, exp_avg, exp_avg_sq, n, lr_dev, beta1, beta2, eps, weight_decay,
                                                       step_dev, world, rank, signal_base, epoch_dev, scratch2_dev + 1, peer_timeout_ns());
    MMS_LAUNCH_CHECK("peer_allreduce_adam_kernel");
    return MMS_OK;
}

extern "C" int mms_peer_allreduce_adam_ranges(float* params, const void* const* grads_host, void* const* signals_host, int32_t world,
                                              int32_t rank, int32_t signal_base, float* exp_avg, float* exp_avg_sq,
                                              const int64_t* ranges_host, int32_t nranges, int64_t* steps_dev, const float* lr_dev,
                                              float beta1, float beta2, float eps, float weight_decay, int64_t* step_dev,
                                              uint32_t* epoch_dev, uint32_t* scratch2_dev, mms_stream_t stream) {
    MMS_REQUIRE(params && grads_host && signals_host && exp_avg && exp_avg_sq && steps_dev && lr_dev && step_dev && epoch_dev &&
                    scratch2_dev && rank >= 0 && rank < world && signal_base >= 0,
                "peer_allreduce_adam_ranges: bad arguments");
    AdamRanges r;
    int rc = adam_ranges_from_host(ranges_host, nranges, INT64_MAX / 2, &r);
    if (rc) return rc;
    PeerPtrs pp;
    rc = fill_peer(&pp, grads_host, signals_host, world);
    if (rc) return rc;
    int64_t n = 0;
    for (int k = 0; k < r.n; ++k) n += r.cnt[k];
    int blocks = (int)((n + 255) / 256);
    if (blocks > 64) blocks = 64;
    if (blocks < 1) blocks = 1;
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    peer_allreduce_adam_ranges_kernel<<<blocks, 256, 0, st>>>(params, pp, exp_avg, exp_avg_sq, r, steps_dev, lr_dev, beta1, beta2, eps,
                                                              weight_decay, step_dev, world, rank, signal_base, epoch_dev,
                                                              scratch2_dev + 1, peer_timeout_ns());
    MMS_LAUNCH_CHECK("peer_allreduce_adam_ranges_kernel");
    return MMS_OK;
}

namespace mms {
int clip_ranges_from_host(const int64_t* ranges_host, int32_t nranges, int64_t n, AdamRanges* r);     // grad_clip.cu
}

extern "C" int mms_peer_grad_norm(const void* const* grads_host, void* const* signals_host, int32_t world, int32_t rank,
                                  int32_t signal_base, int64_t n, const int64_t* ranges_host, int32_t nranges, const float* max_norm,
                                  double* record, void* clip_scratch, uint32_t* norm_epoch_dev, mms_stream_t stream) {
    MMS_REQUIRE(grads_host && signals_host && max_norm && clip_scratch && norm_epoch_dev && rank >= 0 && rank < world && signal_base >= 0,
                "peer_grad_norm: bad arguments");
    MMS_REQUIRE((reinterpret_cast<uintptr_t>(clip_scratch) & 7) == 0, "peer_grad_norm: clip_scratch must be 8-byte aligned");
    AdamRanges r;
    int rc = clip_ranges_from_host(ranges_host, nranges, n, &r);
    if (rc) return rc;
    PeerPtrs pp;
    rc = fill_peer(&pp, grads_host, signals_host, world);
    if (rc) return rc;
    int64_t cnt = 0;
    for (int k = 0; k < r.n; ++k) cnt += r.cnt[k];
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    peer_grad_norm_kernel<<<grad_norm_blocks(cnt), 256, 0, st>>>(pp, world, rank, signal_base, r, max_norm, record,
                                                                 reinterpret_cast<ClipScratch*>(clip_scratch), norm_epoch_dev,
                                                                 peer_timeout_ns());
    MMS_LAUNCH_CHECK("peer_grad_norm_kernel");
    return MMS_OK;
}

extern "C" int mms_peer_allreduce_adam_clip(float* params, const void* const* grads_host, void* const* signals_host, int32_t world,
                                            int32_t rank, int32_t signal_base, float* exp_avg, float* exp_avg_sq, int64_t n,
                                            const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                                            int64_t* step_dev, uint32_t* epoch_dev, uint32_t* scratch2_dev, const float* coef_dev,
                                            mms_stream_t stream) {
    MMS_REQUIRE(params && grads_host && signals_host && exp_avg && exp_avg_sq && lr_dev && step_dev && epoch_dev && scratch2_dev &&
                    coef_dev && rank >= 0 && rank < world && n > 0 && signal_base >= 0,
                "peer_allreduce_adam_clip: bad arguments");
    MMS_REQUIRE(((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(exp_avg) | reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0,
                "peer_allreduce_adam_clip: buffers must be 16-byte aligned");
    PeerPtrs pp;
    int rc = fill_peer(&pp, grads_host, signals_host, world);
    if (rc) return rc;
    for (int i = 0; i < world; ++i)
        MMS_REQUIRE((reinterpret_cast<uintptr_t>(pp.buf[i]) & 15) == 0, "peer_allreduce_adam_clip: gradient buffers must be 16-byte aligned");
    int blocks = (int)((n / 4 + 255) / 256);
    if (blocks > 64) blocks = 64;
    if (blocks < 1) blocks = 1;
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    peer_allreduce_adam_clip_kernel<<<blocks, 256, 0, st>>>(params, pp, exp_avg, exp_avg_sq, n, lr_dev, beta1, beta2, eps, weight_decay,
                                                            step_dev, world, rank, signal_base, epoch_dev, scratch2_dev + 1,
                                                            peer_timeout_ns(), coef_dev);
    MMS_LAUNCH_CHECK("peer_allreduce_adam_clip_kernel");
    return MMS_OK;
}

extern "C" int mms_peer_allreduce_adam_ranges_clip(float* params, const void* const* grads_host, void* const* signals_host, int32_t world,
                                                   int32_t rank, int32_t signal_base, float* exp_avg, float* exp_avg_sq,
                                                   const int64_t* ranges_host, int32_t nranges, int64_t* steps_dev, const float* lr_dev,
                                                   float beta1, float beta2, float eps, float weight_decay, int64_t* step_dev,
                                                   uint32_t* epoch_dev, uint32_t* scratch2_dev, const float* coef_dev,
                                                   mms_stream_t stream) {
    MMS_REQUIRE(params && grads_host && signals_host && exp_avg && exp_avg_sq && steps_dev && lr_dev && step_dev && epoch_dev &&
                    scratch2_dev && coef_dev && rank >= 0 && rank < world && signal_base >= 0,
                "peer_allreduce_adam_ranges_clip: bad arguments");
    AdamRanges r;
    int rc = adam_ranges_from_host(ranges_host, nranges, INT64_MAX / 2, &r);
    if (rc) return rc;
    PeerPtrs pp;
    rc = fill_peer(&pp, grads_host, signals_host, world);
    if (rc) return rc;
    int64_t n = 0;
    for (int k = 0; k < r.n; ++k) n += r.cnt[k];
    int blocks = (int)((n + 255) / 256);
    if (blocks > 64) blocks = 64;
    if (blocks < 1) blocks = 1;
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    peer_allreduce_adam_ranges_clip_kernel<<<blocks, 256, 0, st>>>(params, pp, exp_avg, exp_avg_sq, r, steps_dev, lr_dev, beta1, beta2,
                                                                   eps, weight_decay, step_dev, world, rank, signal_base, epoch_dev,
                                                                   scratch2_dev + 1, peer_timeout_ns(), coef_dev);
    MMS_LAUNCH_CHECK("peer_allreduce_adam_ranges_clip_kernel");
    return MMS_OK;
}
