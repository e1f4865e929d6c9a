// Integrated gradients (attribution.py): the two element-wise passes around each chunk's forward / input-gradient pair.
// A chunk is a run of rows r = b * steps + k (window b, step k) of the B * steps interpolation rows, in order; the
// midpoint rule puts step k at alpha_k = (k + 1/2) / steps.  Every sum over k runs in increasing k inside one thread, and
// chunks are accumulated in row order, so A does not depend on where the chunks are cut (S only to float64 rounding).
#include "mms_common.cuh"

namespace mms {

// z[r] = x0[b] + alpha_k (x[b] - x0[b]),  dlogits[r] = one_hot(target[b]).  grid = (cdiv(n, 1024), nrows), block = 256.
__global__ void __launch_bounds__(256) ig_interpolate_kernel(const float* __restrict__ x, const float* __restrict__ x0,
                                                             int64_t x0_ws, const int64_t* __restrict__ target, int64_t n,
                                                             int steps, int64_t row0, int nc, float* __restrict__ z,
                                                             float* __restrict__ dlogits) {
    const int64_t r = row0 + blockIdx.y;
    const int64_t b = r / steps;
    const int k = (int)(r - b * steps);
    const float alpha = ((float)k + 0.5f) / (float)steps;
    const float* xb = x + b * n;
    const float* x0b = x0 + b * x0_ws;
    float* zr = z + (int64_t)blockIdx.y * n;
    const int64_t e1 = min(n, (int64_t)(blockIdx.x + 1) * 1024);
    for (int64_t e = (int64_t)blockIdx.x * 1024 + threadIdx.x; e < e1; e += blockDim.x) {
        const float base = __ldg(x0b + e);
        zr[e] = base + alpha * (__ldg(xb + e) - base);
    }
    if (blockIdx.x == 0 && threadIdx.x < nc) dlogits[(int64_t)blockIdx.y * nc + threadIdx.x] = target[b] == threadIdx.x ? 1.f : 0.f;
}

// A[b,c,t] += sum_k (x - x0)[b,c,t] dx[r,c,t] / steps and S[b,c] += the same terms summed over t in float64, for the rows
// r in [row0, row0 + nrows).  One CTA per (channel, window of the chunk): no atomics, a fixed reduction order.
// grid = (C, windows touched by the chunk), block = 256.
__global__ void __launch_bounds__(256) ig_accumulate_kernel(const float* __restrict__ x, const float* __restrict__ x0,
                                                            int64_t x0_ws, const float* __restrict__ dx, int C, int T,
                                                            int steps, int64_t row0, int nrows, float* __restrict__ A,
                                                            double* __restrict__ S) {
    __shared__ double s_part[8];
    const int c = blockIdx.x;
    const int64_t b = row0 / steps + blockIdx.y;
    const int64_t n = (int64_t)C * T;
    const int k0 = (int)max((int64_t)0, row0 - b * steps);
    const int k1 = (int)min((int64_t)steps, row0 + nrows - b * steps);
    const float inv_m = 1.f / (float)steps;
    const float* xr = x + b * n + (int64_t)c * T;
    const float* x0r = x0 + b * x0_ws + (int64_t)c * T;
    const float* dxr = dx + (b * steps + k0 - row0) * n + (int64_t)c * T;
    float* Ar = A + b * n + (int64_t)c * T;
    double s = 0.0;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        const float diff = __ldg(xr + t) - __ldg(x0r + t);
        float a = Ar[t];
        for (int k = k0; k < k1; ++k) {
            const float v = diff * __ldg(dxr + (int64_t)(k - k0) * n + t) * inv_m;
            a += v;
            s += (double)v;
        }
        Ar[t] = a;
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < 8; ++w) tot += s_part[w];
        S[b * C + c] += tot;
    }
}

}  // namespace mms

using namespace mms;

extern "C" int mms_ig_interpolate(const float* x, const float* x0, int32_t x0_per_window, const int64_t* target, int32_t B,
                                  int32_t C, int32_t T, int32_t num_classes, int32_t steps, int64_t row0, int32_t nrows, float* z,
                                  float* dlogits, mms_stream_t stream) {
    MMS_REQUIRE(x && x0 && target && z && dlogits, "ig_interpolate: null pointer");
    MMS_REQUIRE(B >= 1 && C >= 1 && T >= 1 && steps >= 1 && num_classes >= 1 && num_classes <= 256, "ig_interpolate: bad sizes");
    MMS_REQUIRE(row0 >= 0 && nrows >= 1 && nrows <= 65535 && row0 + nrows <= (int64_t)B * steps, "ig_interpolate: rows outside [0, B*steps)");
    const int64_t n = (int64_t)C * T;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(cdiv(n, 1024), nrows);
    MMS_PROF_BEGIN(st);
    ig_interpolate_kernel<<<grid, 256, 0, st>>>(x, x0, x0_per_window ? n : 0, target, n, steps, row0, num_classes, z, dlogits);
    MMS_LAUNCH_CHECK("ig_interpolate_kernel");
    return MMS_OK;
}

extern "C" int mms_ig_accumulate(const float* x, const float* x0, int32_t x0_per_window, const float* dx, int32_t B, int32_t C,
                                 int32_t T, int32_t steps, int64_t row0, int32_t nrows, float* A, double* S, mms_stream_t stream) {
    MMS_REQUIRE(x && x0 && dx && A && S, "ig_accumulate: null pointer");
    MMS_REQUIRE(B >= 1 && C >= 1 && T >= 1 && steps >= 1, "ig_accumulate: bad sizes");
    MMS_REQUIRE(row0 >= 0 && nrows >= 1 && row0 + nrows <= (int64_t)B * steps, "ig_accumulate: rows outside [0, B*steps)");
    const int64_t nwin = (row0 + nrows - 1) / steps - row0 / steps + 1;
    MMS_REQUIRE(nwin <= 65535, "ig_accumulate: %lld windows in one chunk", (long long)nwin);
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(C, (unsigned)nwin);
    MMS_PROF_BEGIN(st);
    ig_accumulate_kernel<<<grid, 256, 0, st>>>(x, x0, x0_per_window ? (int64_t)C * T : 0, dx, C, T, steps, row0, nrows, A, S);
    MMS_LAUNCH_CHECK("ig_accumulate_kernel");
    return MMS_OK;
}
