// Gradient-norm clipping (torch.nn.utils.clip_grad_norm_, norm_type 2) between the backward and Adam: the norm kernel and the
// clipped forms of adam_flat_kernel / adam_ranges_kernel (head_opt.cu).  Those two stay as they are: the clipped update is a
// separate pair of kernels that read the coefficient the norm kernel wrote, so a step without clipping runs exactly the code it
// ran before.  The device helpers (ClipScratch, grad_norm_finish, clip_coef, adam_update_clipped) are in mms_common.cuh; the
// peer-path kernels in peer.cu.
#include "mms_common.cuh"

namespace mms {

// Sum of squares (float64, of the fp32 values) over the virtual index space of `r`, then grad_norm_finish.
__global__ void __launch_bounds__(256) grad_norm_kernel(const float* __restrict__ g, const __grid_constant__ AdamRanges r,
                                                        const float* __restrict__ max_norm_dev, double* record, ClipScratch* cs) {
    MMS_PDL_PROLOGUE();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double s = 0.0;
    int64_t base = 0;
    for (int k = 0; k < r.n; ++k) {
        int64_t j = (gt - base) % stride;
        if (j < 0) j += stride;
        const float* gk = g + r.off[k];
        for (; j < r.cnt[k]; j += stride) {
            const double x = (double)gk[j];
            s += x * x;
        }
        base += r.cnt[k];
    }
    grad_norm_finish(s, cs, max_norm_dev, record);
}

// adam_flat_kernel on coef * g
__global__ void __launch_bounds__(256) adam_flat_clip_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                             float* __restrict__ v, int64_t n, const float* __restrict__ lr_dev,
                                                             float beta1, float beta2, float eps, float wd, int64_t* step_dev,
                                                             int32_t* scratch, const float* __restrict__ coef_dev) {
    MMS_PDL_PROLOGUE();
    const int64_t done = *step_dev;
    const float lr = *lr_dev;
    const float coef = *coef_dev;
    const AdamCoef c = adam_coef(done, lr, beta1, beta2);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        adam_update_clipped(p, g, m, v, i, coef, c, beta1, beta2, eps, wd);
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const int last = atomicAdd(scratch, 1);
        if (last == (int)gridDim.x - 1) {
            *step_dev += 1;
            *scratch = 0;
        }
    }
}

// adam_ranges_kernel on coef * g
__global__ void __launch_bounds__(256) adam_ranges_clip_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                               float* __restrict__ v, const __grid_constant__ AdamRanges r,
                                                               int64_t* steps, const float* __restrict__ lr_dev, float beta1,
                                                               float beta2, float eps, float wd, int64_t* step_dev, int32_t* scratch,
                                                               const float* __restrict__ coef_dev) {
    MMS_PDL_PROLOGUE();
    __shared__ AdamCoef s_c[MMS_MAX_ADAM_RANGES];
    const float lr = *lr_dev;
    for (int k = threadIdx.x; k < r.n; k += blockDim.x) s_c[k] = adam_coef(steps[r.slot[k]], lr, beta1, beta2);
    __syncthreads();
    const float coef = *coef_dev;            // read after the pow() calls above: live across them it costs a spill
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t base = 0;
    for (int k = 0; k < r.n; ++k) {
        const AdamCoef c = s_c[k];
        int64_t j = (gt - base) % stride;
        if (j < 0) j += stride;
        for (; j < r.cnt[k]; j += stride) adam_update_clipped(p, g, m, v, r.off[k] + j, coef, c, beta1, beta2, eps, wd);
        base += r.cnt[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const int done = atomicAdd(scratch, 1);
        if (done == (int)gridDim.x - 1) {
            for (int k = 0; k < r.n; ++k) steps[r.slot[k]] += 1;
            *step_dev += 1;
            *scratch = 0;
        }
    }
}

int launch_grad_norm(const float* g, const AdamRanges& r, const float* max_norm_dev, double* record, void* clip_scratch,
                     cudaStream_t st) {
    MMS_REQUIRE(g && max_norm_dev && clip_scratch, "grad_norm: null pointer");
    MMS_REQUIRE((reinterpret_cast<uintptr_t>(clip_scratch) & 7) == 0, "grad_norm: clip_scratch must be 8-byte aligned");
    int64_t n = 0;
    for (int k = 0; k < r.n; ++k) n += r.cnt[k];
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(grad_norm_kernel, dim3(grad_norm_blocks(n)), dim3(256), 0, st, g, r, max_norm_dev, record,
               reinterpret_cast<ClipScratch*>(clip_scratch));
    MMS_LAUNCH_CHECK("grad_norm_kernel");
    return MMS_OK;
}

// The grid sizes of launch_adam / launch_adam_ranges (head_opt.cu), so that coef == 1 reproduces them bit for bit.
int launch_adam_clip(float* p, const float* g, float* m, float* v, int64_t n, const float* lr_dev, float beta1, float beta2,
                     float eps, float wd, int64_t* step_dev, int32_t* scratch, const float* coef_dev, cudaStream_t st) {
    const int blocks = (int)((n + 255) / 256 < 592 ? (n + 255) / 256 : 592);
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(adam_flat_clip_kernel, dim3(blocks > 0 ? blocks : 1), dim3(256), 0, st, p, g, m, v, n, lr_dev, beta1, beta2, eps, wd,
               step_dev, scratch, coef_dev);
    MMS_LAUNCH_CHECK("adam_flat_clip_kernel");
    return MMS_OK;
}

int launch_adam_ranges_clip(float* p, const float* g, float* m, float* v, const AdamRanges& r, int64_t* steps, const float* lr_dev,
                            float beta1, float beta2, float eps, float wd, int64_t* step_dev, int32_t* scratch, const float* coef_dev,
                            cudaStream_t st) {
    int64_t n = 0;
    for (int k = 0; k < r.n; ++k) n += r.cnt[k];
    const int blocks = (int)((n + 255) / 256 < 592 ? (n + 255) / 256 : 592);
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(adam_ranges_clip_kernel, dim3(blocks > 0 ? blocks : 1), dim3(256), 0, st, p, g, m, v, r, steps, lr_dev, beta1, beta2,
               eps, wd, step_dev, scratch, coef_dev);
    MMS_LAUNCH_CHECK("adam_ranges_clip_kernel");
    return MMS_OK;
}

// ranges_host (HOST (offset, count, slot) rows) or, when NULL, the single range [0, n)
int clip_ranges_from_host(const int64_t* ranges_host, int32_t nranges, int64_t n, AdamRanges* r) {
    if (ranges_host) return adam_ranges_from_host(ranges_host, nranges, INT64_MAX / 2, r);
    MMS_REQUIRE(n > 0 && nranges == 0, "grad_norm: without a range table n must be > 0 and nranges 0");
    r->n = 1;
    r->off[0] = 0;
    r->cnt[0] = n;
    r->slot[0] = 0;
    return MMS_OK;
}

}  // namespace mms

using namespace mms;

extern "C" int mms_grad_norm(const float* grads, int64_t n, const int64_t* ranges_host, int32_t nranges, const float* max_norm,
                             double* record, void* clip_scratch, mms_stream_t stream) {
    AdamRanges r;
    const int rc = clip_ranges_from_host(ranges_host, nranges, n, &r);
    if (rc) return rc;
    return launch_grad_norm(grads, r, max_norm, record, clip_scratch, (cudaStream_t)stream);
}

extern "C" int mms_adam_flat_clip_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                                       const float* lr_dev, float beta1, float beta2, float eps, float weight_decay, int64_t* step_dev,
                                       int32_t* scratch_dev, const float* coef_dev, mms_stream_t stream) {
    MMS_REQUIRE(params && grads && exp_avg && exp_avg_sq && lr_dev && step_dev && scratch_dev && coef_dev && n > 0,
                "adam_flat_clip_step: bad arguments");
    return launch_adam_clip(params, grads, exp_avg, exp_avg_sq, n, lr_dev, beta1, beta2, eps, weight_decay, step_dev, scratch_dev,
                            coef_dev, (cudaStream_t)stream);
}

extern "C" int mms_adam_ranges_clip_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                                         const int64_t* ranges_host, int32_t nranges, int64_t* steps_dev, const float* lr_dev,
                                         float beta1, float beta2, float eps, float weight_decay, int64_t* step_dev,
                                         int32_t* scratch_dev, const float* coef_dev, mms_stream_t stream) {
    MMS_REQUIRE(params && grads && exp_avg && exp_avg_sq && steps_dev && lr_dev && step_dev && scratch_dev && coef_dev,
                "adam_ranges_clip_step: bad arguments");
    AdamRanges r;
    const int rc = adam_ranges_from_host(ranges_host, nranges, INT64_MAX / 2, &r);
    if (rc) return rc;
    return launch_adam_ranges_clip(params, grads, exp_avg, exp_avg_sq, r, steps_dev, lr_dev, beta1, beta2, eps, weight_decay, step_dev,
                                   scratch_dev, coef_dev, (cudaStream_t)stream);
}
