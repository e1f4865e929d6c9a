// Monte-Carlo dropout (uncertainty.py, mms_cnngru_mc_forward in model.cu): the two element-wise kernels around the shared
// prefix and the per-sample layers.  Sample s of window b is sample row r = b * samples + s; a chunk is the sample rows
// [row0, row0 + nrows) and every multiplier is drawn with the global row r (oracle/dropout_stream.py, "MC sampling").
#include "mms_common.cuh"

namespace mms {

constexpr int MC_MAX_NC = 8;

// out[r, k] = src[r / samples, k] * mult(drop_base + r * row_len + k) for the nrows sample rows of a chunk, which starts at
// a window boundary; the source row of the chunk's window w starts at src + w * src_ld.  drop_base already holds the
// chunk's first row (site base + row0 * row_len); p == 0 copies.  row_len % 4 == 0 and 16-byte aligned rows: one float4 per
// thread and step.
__global__ void __launch_bounds__(256) mc_expand_kernel(const float* __restrict__ src, int64_t src_ld, int64_t row_len,
                                                        int samples, int64_t nrows, float* __restrict__ out, int64_t drop_base,
                                                        float p, uint64_t seed, uint64_t offset, const int64_t* offset_dev) {
    DropRng rng;
    if (p > 0.f) rng.init(seed, resolve_offset(offset, offset_dev), p);
    const int64_t q = row_len >> 2, n4 = nrows * q;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const int64_t r = i / q, k = 4 * (i - r * q);
        float4 v = __ldg(reinterpret_cast<const float4*>(src + (r / samples) * src_ld + k));
        if (p > 0.f) {
            const uint64_t e = (uint64_t)(drop_base + r * row_len + k);
            v.x *= rng.mult(e); v.y *= rng.mult(e + 1); v.z *= rng.mult(e + 2); v.w *= rng.mult(e + 3);
        }
        reinterpret_cast<float4*>(out)[i] = v;
    }
}

// One thread per window the chunk touches: for its rows in increasing s it adds, in float64, the softmax p_s of the
// logits to psum[b, :] and the entropy -sum p_s log p_s (0 log 0 = 0) to hsum[b]; the thread that adds a window's last
// sample writes probs = psum / samples, entropy = H(probs) and mutual_info = entropy - hsum / samples.  Chunks are
// accumulated in row order, so every window sees the same sequence of additions however the rows are chunked.
__global__ void __launch_bounds__(128) mc_accumulate_kernel(const float* __restrict__ logits, int nc, int samples, int64_t row0,
                                                            int nrows, int nwin, double* __restrict__ psum,
                                                            double* __restrict__ hsum, double* __restrict__ probs,
                                                            double* __restrict__ entropy, double* __restrict__ mutual_info) {
    const int wi = blockIdx.x * blockDim.x + threadIdx.x;
    if (wi >= nwin) return;
    const int64_t b = row0 / samples + wi;
    const int64_t r0 = max(row0, b * samples), r1 = min(row0 + nrows, (b + 1) * samples);
    double ps[MC_MAX_NC];
#pragma unroll
    for (int c = 0; c < MC_MAX_NC; ++c) ps[c] = c < nc ? psum[b * nc + c] : 0.0;
    double hs = hsum[b];
    for (int64_t r = r0; r < r1; ++r) {
        const float* l = logits + (r - row0) * nc;
        double v[MC_MAX_NC], mx = -INFINITY, se = 0.0;
#pragma unroll
        for (int c = 0; c < MC_MAX_NC; ++c)
            if (c < nc) { v[c] = (double)l[c]; mx = fmax(mx, v[c]); }
#pragma unroll
        for (int c = 0; c < MC_MAX_NC; ++c)
            if (c < nc) { v[c] = exp(v[c] - mx); se += v[c]; }
        double h = 0.0;
#pragma unroll
        for (int c = 0; c < MC_MAX_NC; ++c)
            if (c < nc) {
                const double pc = v[c] / se;
                ps[c] += pc;
                if (pc > 0.0) h -= pc * log(pc);
            }
        hs += h;
    }
#pragma unroll
    for (int c = 0; c < MC_MAX_NC; ++c)
        if (c < nc) psum[b * nc + c] = ps[c];
    hsum[b] = hs;
    if (r1 == (b + 1) * samples) {
        double ent = 0.0;
#pragma unroll
        for (int c = 0; c < MC_MAX_NC; ++c)
            if (c < nc) {
                const double pm = ps[c] / samples;
                probs[b * nc + c] = pm;
                if (pm > 0.0) ent -= pm * log(pm);
            }
        entropy[b] = ent;
        mutual_info[b] = ent - hs / samples;
    }
}

int launch_mc_expand(const float* src, int64_t src_ld, int64_t row_len, int samples, int64_t nrows, float* out, int64_t drop_base,
                     float p, uint64_t seed, uint64_t offset, const int64_t* offset_dev, cudaStream_t st) {
    MMS_REQUIRE(src && out && samples >= 1 && nrows >= 1 && row_len >= 4, "mc_expand: bad arguments");
    MMS_REQUIRE(row_len % 4 == 0 && src_ld % 4 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(out)) & 15) == 0,
                "mc_expand: rows must be 16-byte aligned multiples of 4 floats");
    int64_t blocks = (nrows * (row_len / 4) + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    MMS_PROF_BEGIN(st);
    mc_expand_kernel<<<(int)blocks, 256, 0, st>>>(src, src_ld, row_len, samples, nrows, out, drop_base, p, seed, offset, offset_dev);
    MMS_LAUNCH_CHECK("mc_expand_kernel");
    return MMS_OK;
}

}  // namespace mms

using namespace mms;

extern "C" int mms_mc_accumulate(const float* logits, int32_t B, int32_t nc, int32_t samples, int64_t row0, int32_t nrows,
                                 double* psum, double* hsum, double* probs, double* entropy, double* mutual_info,
                                 mms_stream_t stream) {
    MMS_REQUIRE(logits && psum && hsum && probs && entropy && mutual_info, "mc_accumulate: null pointer");
    MMS_REQUIRE(B >= 1 && samples >= 1 && nc >= 1 && nc <= MC_MAX_NC, "mc_accumulate: bad sizes");
    MMS_REQUIRE(row0 >= 0 && nrows >= 1 && row0 + nrows <= (int64_t)B * samples, "mc_accumulate: rows outside [0, B*samples)");
    const int64_t nwin = (row0 + nrows - 1) / samples - row0 / samples + 1;
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    mc_accumulate_kernel<<<(unsigned)cdiv(nwin, 128), 128, 0, st>>>(logits, nc, samples, row0, nrows, (int)nwin, psum, hsum, probs,
                                                                    entropy, mutual_info);
    MMS_LAUNCH_CHECK("mc_accumulate_kernel");
    return MMS_OK;
}
