// Classifier head (reference models.py:66-71,79-80), CrossEntropyLoss (trainer.py:69,147; optionally class-weighted, trainer.py:94) and the
// fused flat Adam (trainer.py:68,149).  All tiny, latency-bound kernels: the point of fusing them is
// launch count, not bandwidth.
#include "mms_common.cuh"

namespace mms {

constexpr int MAX_NC = 8;
constexpr uint64_t HEAD_DROP_BASE = 0x4000000000ull;   // element ids of the head dropout site

// grid = B, block = 4 * 64: thread (i, q) = (tid >> 2, tid & 3) sums a quarter of hidden unit i's dot product (128-bit
// weight loads, all in flight at once) and the four quarters meet by shuffles.  hid_out keeps relu(W0 last + b0)
// (before dropout).  The classifier input is the concatenation [src_a[b, 0:Hh) | src_b[b, 0:H2-Hh)] (forward-direction
// final state and reverse-direction first-step state, models.py:79); it is also written to last_out.  Row b draws its
// dropout multipliers as row drop_row0 + b of the head site (0 for a whole batch; MC dropout passes its chunk's first
// sample row).
__global__ void __launch_bounds__(4 * HEAD_HID) head_fwd_kernel(const float* __restrict__ src_a, int64_t lda,
                                                                const float* __restrict__ src_b, int64_t ldb, int Hh,
                                                                const float* __restrict__ w0,
                                                                const float* __restrict__ b0, const float* __restrict__ w3,
                                                                const float* __restrict__ b3, int H2, int nc, float p,
                                                                uint64_t seed, uint64_t offset, const int64_t* offset_dev,
                                                                int64_t drop_row0, float* __restrict__ last_out,
                                                                float* __restrict__ hid_out, float* __restrict__ logits) {
    MMS_PDL_PROLOGUE();
    extern __shared__ __align__(16) float s_last[];        // [H2]
    __shared__ float s_hid[HEAD_HID];
    const int b = blockIdx.x, tid = threadIdx.x, i = tid >> 2, q = tid & 3;
    for (int k = tid; k < H2; k += 4 * HEAD_HID) {
        const float v = k < Hh ? src_a[(size_t)b * lda + k] : src_b[(size_t)b * ldb + (k - Hh)];
        s_last[k] = v;
        if (last_out) last_out[(size_t)b * H2 + k] = v;
    }
    __syncthreads();
    float acc = 0.f;
    const float* wr = w0 + (size_t)i * H2;
    if ((H2 & 15) == 0 && (reinterpret_cast<uintptr_t>(w0) & 15) == 0) {
        const int kq = H2 >> 2;                            // this lane's quarter [q*kq, (q+1)*kq), a multiple of 4
        const float4* w4 = reinterpret_cast<const float4*>(wr + q * kq);
        const float4* l4 = reinterpret_cast<const float4*>(s_last + q * kq);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
        for (int k4 = 0; k4 < (kq >> 2); ++k4) {
            const float4 wv = __ldg(w4 + k4), lv = l4[k4];
            a0 = fmaf(wv.x, lv.x, a0); a1 = fmaf(wv.y, lv.y, a1); a2 = fmaf(wv.z, lv.z, a2); a3 = fmaf(wv.w, lv.w, a3);
        }
        acc = (a0 + a1) + (a2 + a3);
    } else {
        for (int k = q; k < H2; k += 4) acc = fmaf(__ldg(wr + k), s_last[k], acc);
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    if (q == 0) {
        const float h = fmaxf(acc + b0[i], 0.f);
        hid_out[(size_t)b * HEAD_HID + i] = h;
        float m = 1.f;
        if (p > 0.f) {
            DropRng rng;
            rng.init(seed, resolve_offset(offset, offset_dev), p);
            m = rng.mult(HEAD_DROP_BASE + (uint64_t)(drop_row0 + b) * HEAD_HID + i);
        }
        s_hid[i] = h * m;
    }
    __syncthreads();
    if (tid < nc) {
        float l = b3[tid];
        for (int k = 0; k < HEAD_HID; ++k) l = fmaf(w3[tid * HEAD_HID + k], s_hid[k], l);
        logits[(size_t)b * nc + tid] = l;
    }
}

// Training-step fusion of head forward + CrossEntropyLoss + the head's input-side backward (reference models.py:79-80,
// trainer.py:147-148): ONE launch on the step's critical path instead of three (head_fwd, cross_entropy, head_bwd).  grid = B,
// block = 4 * 64, same thread mapping as head_fwd_kernel.  Row b's CTA computes hid, logits, its loss term
// lse - logit[y], dlogits = (softmax - onehot) / div_batch and dhid = relu'(hid) * mask * (W3^T dlogits) -- everything the
// top-layer GRU backward needs (it multiplies dhid by W0 itself).  The weight gradients of the head do not feed the chain:
// head_bwd_kernel computes them on a side stream (dhid = nullptr there: no second write).  The mean loss is formed by the
// LAST CTA to finish (counter zeroed with the forward's memset) from the per-row terms in a fixed order, so the loss is
// bit-reproducible run to run.  Labels outside [0, nc) poison the loss with NaN (torch raises; a silent clamp would train on
// garbage) and contribute no gradient.
// class_weight (optional, [nc]): CrossEntropyLoss(weight=w).  Every CTA needs the normaliser W = sum_b w[y_b] before it can
// write dlogits; rather than wait on the other CTAs, each one reduces the B labels itself (warp 1, while the other warps load
// the classifier input), in the same fixed order, so all CTAs hold the same bit pattern.  The row term becomes w[y]*(lse - logit[y]),
// dlogits (softmax - onehot) * w[y] / W and the loss sum_b w*l / W.  The host picks the instance by the pointer: with the
// weighted code compiled out, a null pointer runs exactly the unweighted kernel (an in-kernel branch on the pointer measured
// ~1 us slower per training step on a B200 with weights off: a larger kernel scheduled differently).
template <bool WEIGHTED>
__global__ void __launch_bounds__(4 * HEAD_HID) head_ce_fused_kernel(const float* __restrict__ src_a, int64_t lda,
                                                                     const float* __restrict__ src_b, int64_t ldb, int Hh,
                                                                     const float* __restrict__ w0, const float* __restrict__ b0,
                                                                     const float* __restrict__ w3, const float* __restrict__ b3,
                                                                     const int64_t* __restrict__ labels, int H2, int nc, float p,
                                                                     uint64_t seed, uint64_t offset, const int64_t* offset_dev,
                                                                     int div_batch, float* __restrict__ last_out,
                                                                     float* __restrict__ hid_out, float* __restrict__ logits,
                                                                     float* __restrict__ dlogits, float* __restrict__ dhid,
                                                                     float* __restrict__ rowloss, int32_t* __restrict__ counter,
                                                                     float* __restrict__ loss_out, double* __restrict__ loss_sum_accum,
                                                                     const float* __restrict__ class_weight) {
    MMS_PDL_PROLOGUE();
    extern __shared__ __align__(16) float s_last[];        // [H2]
    __shared__ float s_hid[HEAD_HID], s_mask[HEAD_HID], s_logit[MAX_NC], s_dl[MAX_NC];
    __shared__ int s_last_cta;
    __shared__ float s_wsum;
    const int b = blockIdx.x, B = gridDim.x, tid = threadIdx.x, i = tid >> 2, q = tid & 3;
    if (WEIGHTED && (tid >> 5) == 1) {
        const int lane = tid & 31;
        double ws = 0.0;
        for (int r = lane; r < B; r += 32) {
            const int64_t yr = labels[r];
            if (yr >= 0 && yr < nc) ws += (double)__ldg(class_weight + yr);
        }
        ws = warp_sum(ws);
        if (lane == 0) s_wsum = (float)ws;
    }
    for (int k = tid; k < H2; k += 4 * HEAD_HID) {
        const float v = k < Hh ? src_a[(size_t)b * lda + k] : src_b[(size_t)b * ldb + (k - Hh)];
        s_last[k] = v;
        last_out[(size_t)b * H2 + k] = v;
    }
    __syncthreads();
    float acc = 0.f;
    const float* wr = w0 + (size_t)i * H2;
    if ((H2 & 15) == 0 && (reinterpret_cast<uintptr_t>(w0) & 15) == 0) {
        const int kq = H2 >> 2;
        const float4* w4 = reinterpret_cast<const float4*>(wr + q * kq);
        const float4* l4 = reinterpret_cast<const float4*>(s_last + q * kq);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
        for (int k4 = 0; k4 < (kq >> 2); ++k4) {
            const float4 wv = __ldg(w4 + k4), lv = l4[k4];
            a0 = fmaf(wv.x, lv.x, a0); a1 = fmaf(wv.y, lv.y, a1); a2 = fmaf(wv.z, lv.z, a2); a3 = fmaf(wv.w, lv.w, a3);
        }
        acc = (a0 + a1) + (a2 + a3);
    } else {
        for (int k = q; k < H2; k += 4) acc = fmaf(__ldg(wr + k), s_last[k], acc);
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    float h = 0.f, m = 1.f;
    if (q == 0) {
        h = fmaxf(acc + b0[i], 0.f);
        hid_out[(size_t)b * HEAD_HID + i] = h;
        if (p > 0.f) {
            DropRng rng;
            rng.init(seed, resolve_offset(offset, offset_dev), p);
            m = rng.mult(HEAD_DROP_BASE + (uint64_t)b * HEAD_HID + i);
        }
        s_hid[i] = h * m;
        s_mask[i] = h > 0.f ? m : 0.f;                      // relu'(hid) * dropout multiplier
    }
    __syncthreads();
    if (tid < nc) {
        float l = b3[tid];
        for (int k = 0; k < HEAD_HID; ++k) l = fmaf(w3[tid * HEAD_HID + k], s_hid[k], l);
        logits[(size_t)b * nc + tid] = l;
        s_logit[tid] = l;
    }
    __syncthreads();
    if (tid == 0) {
        float mx = -INFINITY;
        for (int c = 0; c < nc; ++c) mx = fmaxf(mx, s_logit[c]);
        float se = 0.f;
        for (int c = 0; c < nc; ++c) se += expf(s_logit[c] - mx);
        const float lse = mx + logf(se);
        const int64_t y = labels[b];
        const bool ok = y >= 0 && y < nc;
        float invB, wy = 1.f;
        if (WEIGHTED) {
            wy = ok ? __ldg(class_weight + y) : 0.f;
            invB = wy / s_wsum;
        } else {
            invB = 1.f / (float)div_batch;
        }
        for (int c = 0; c < nc; ++c) {
            const float dl = ok ? (expf(s_logit[c] - lse) - (c == (int)y ? 1.f : 0.f)) * invB : 0.f;
            s_dl[c] = dl;
            dlogits[(size_t)b * nc + c] = dl;
        }
        const float term = ok ? lse - s_logit[(int)y] : __int_as_float(0x7fc00000);
        rowloss[b] = WEIGHTED ? wy * term : term;
        __threadfence();
        s_last_cta = atomicAdd(counter, 1) == B - 1;
    }
    __syncthreads();
    if (tid < HEAD_HID) {
        float dhd = 0.f;
        for (int c = 0; c < nc; ++c) dhd = fmaf(s_dl[c], w3[c * HEAD_HID + tid], dhd);
        dhid[(size_t)b * HEAD_HID + tid] = dhd * s_mask[tid];
    }
    if (s_last_cta && tid < 32) {
        __threadfence();
        float s = 0.f;
        for (int r = tid; r < B; r += 32) s += __ldcg(rowloss + r);       // fixed order: lane-strided sums, then the shuffle tree
        s = warp_sum(s);
        if (tid == 0) {
            const float mean = s / (WEIGHTED ? s_wsum : (float)div_batch);
            loss_out[0] = mean;
            if (loss_sum_accum) *loss_sum_accum += (double)mean * (double)div_batch;
        }
    }
}

// grid = 64 (hidden unit i), block = 128.  Dynamic smem: B floats.
__global__ void __launch_bounds__(128) head_bwd_kernel(const float* __restrict__ last, const float* __restrict__ hid,
                                                       const float* __restrict__ dlogits, const float* __restrict__ w3, int B,
                                                       int H2, int nc, float p, uint64_t seed, uint64_t offset,
                                                       const int64_t* offset_dev, float* __restrict__ dhid,
                                                       float* __restrict__ dw0, float* __restrict__ db0,
                                                       float* __restrict__ dw3, float* __restrict__ db3) {
    MMS_PDL_PROLOGUE();
    extern __shared__ float s_dh[];          // [B]
    __shared__ float s_red[4][MAX_NC + 1];
    const int i = blockIdx.x, tid = threadIdx.x;
    DropRng rng;
    if (p > 0.f) rng.init(seed, resolve_offset(offset, offset_dev), p);
    float w3c[MAX_NC];
#pragma unroll
    for (int c = 0; c < MAX_NC; ++c) w3c[c] = c < nc ? w3[c * HEAD_HID + i] : 0.f;
    float part[MAX_NC + 1];
#pragma unroll
    for (int c = 0; c <= MAX_NC; ++c) part[c] = 0.f;
    for (int b = tid; b < B; b += 128) {
        const float h = hid[(size_t)b * HEAD_HID + i];
        const float m = p > 0.f ? rng.mult(HEAD_DROP_BASE + (uint64_t)b * HEAD_HID + i) : 1.f;
        float dhd = 0.f;
#pragma unroll
        for (int c = 0; c < MAX_NC; ++c)
            if (c < nc) {
                const float dl = dlogits[(size_t)b * nc + c];
                dhd = fmaf(dl, w3c[c], dhd);
                part[c] = fmaf(dl, h * m, part[c]);          // dW3[c,i]
            }
        const float dh = h > 0.f ? dhd * m : 0.f;
        s_dh[b] = dh;
        if (dhid) dhid[(size_t)b * HEAD_HID + i] = dh;
        part[MAX_NC] += dh;                                  // db0[i]
    }
    const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
    for (int c = 0; c <= MAX_NC; ++c) {
        const float v = warp_sum(part[c]);
        if (lane == 0) s_red[warp][c] = v;
    }
    __syncthreads();
    if (tid <= MAX_NC) {
        const float v = s_red[0][tid] + s_red[1][tid] + s_red[2][tid] + s_red[3][tid];
        if (tid < nc) dw3[tid * HEAD_HID + i] += v;
        if (tid == MAX_NC) db0[i] += v;
    }
    for (int k = tid; k < H2; k += 128) {
        float s = 0.f;
        for (int b = 0; b < B; ++b) s = fmaf(s_dh[b], __ldg(last + (size_t)b * H2 + k), s);
        dw0[(size_t)i * H2 + k] += s;
    }
    if (i == 0 && tid < nc) {
        float s = 0.f;
        for (int b = 0; b < B; ++b) s += dlogits[(size_t)b * nc + tid];
        db3[tid] += s;
    }
}

// Single CTA.  loss_out[0] = mean_b(lse_b - logit[b, y_b]); dlogits = (softmax - onehot) / B.
// With class_weight [nc] (CrossEntropyLoss(weight=w)): loss_out[0] = sum_b w[y_b] l_b / W, dlogits = w[y_b] (softmax - onehot) / W,
// where W is *norm (float64, e.g. the global sum under data parallelism) or, with norm == NULL, sum_b w[y_b] over this batch,
// reduced first in a fixed order.  A null class_weight runs exactly the unweighted arithmetic.
__global__ void __launch_bounds__(256) cross_entropy_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                                                            int B, int nc, float* __restrict__ loss_out,
                                                            float* __restrict__ dlogits, double* __restrict__ loss_sum_accum,
                                                            int div_batch, const float* __restrict__ class_weight,
                                                            const double* __restrict__ norm) {
    MMS_PDL_PROLOGUE();
    __shared__ float s_part[8];
    __shared__ double s_wpart[8];
    float local = 0.f;
    float invB = 1.f / (float)div_batch;           // global batch under data parallelism: the per-rank losses add up
    if (class_weight) {
        double W;
        if (norm) {
            W = *norm;
        } else {
            double ws = 0.0;
            for (int b = threadIdx.x; b < B; b += blockDim.x) {
                const int64_t yl = labels[b];
                if (yl >= 0 && yl < nc) ws += (double)class_weight[yl];
            }
            ws = warp_sum(ws);
            if ((threadIdx.x & 31) == 0) s_wpart[threadIdx.x >> 5] = ws;
            __syncthreads();
            W = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) W += s_wpart[w];
        }
        invB = 1.f / (float)W;
    }
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        float v[MAX_NC];
        float mx = -INFINITY;
        for (int c = 0; c < nc; ++c) { v[c] = logits[(size_t)b * nc + c]; mx = fmaxf(mx, v[c]); }
        float se = 0.f;
        for (int c = 0; c < nc; ++c) se += expf(v[c] - mx);
        const float lse = mx + logf(se);
        const int64_t yl = labels[b];
        const bool ok = yl >= 0 && yl < nc;      // torch raises on such a label; here the loss turns NaN and the row adds no gradient
        const int y = ok ? (int)yl : 0;
        if (class_weight) {
            const float wy = ok ? class_weight[y] : 0.f;
            local += ok ? wy * (lse - v[y]) : __int_as_float(0x7fc00000);
            const float scale = wy * invB;
            if (dlogits)
                for (int c = 0; c < nc; ++c) dlogits[(size_t)b * nc + c] = ok ? (expf(v[c] - lse) - (c == y ? 1.f : 0.f)) * scale : 0.f;
            continue;
        }
        local += ok ? lse - v[y] : __int_as_float(0x7fc00000);
        if (dlogits)
            for (int c = 0; c < nc; ++c) dlogits[(size_t)b * nc + c] = ok ? (expf(v[c] - lse) - (c == y ? 1.f : 0.f)) * invB : 0.f;
    }
    local = warp_sum(local);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int w = 0; w < (blockDim.x >> 5); ++w) s += s_part[w];
        const float mean = s * invB;
        loss_out[0] = mean;
        if (loss_sum_accum) *loss_sum_accum += (double)mean * (double)div_batch;
    }
}

// torch.optim.Adam (adam_update, mms_common.cuh) over the flat buffer, t = *step_dev + 1.
// The last CTA to finish increments *step_dev (every CTA has read it by then).
__global__ void __launch_bounds__(256) adam_flat_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                        float* __restrict__ v, int64_t n, const float* __restrict__ lr_dev,
                                                        float beta1, float beta2, float eps, float wd, int64_t* step_dev,
                                                        int32_t* scratch) {
    MMS_PDL_PROLOGUE();
    const int64_t done = *step_dev;
    const float lr = *lr_dev;
    const AdamCoef c = adam_coef(done, lr, beta1, beta2);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        adam_update(p, g, m, v, i, c, beta1, beta2, eps, wd);
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

// The same update over the ranges of `r` only, range k with its own count steps[r.slot[k]].  The ranges are laid end to end
// into one virtual index space that the grid strides over, so small tensors do not all land on the first threads.  The last
// CTA to finish advances every range's count and *step_dev.
__global__ void __launch_bounds__(256) adam_ranges_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                          float* __restrict__ v, const __grid_constant__ AdamRanges r,
                                                          int64_t* steps, const float* __restrict__ lr_dev, float beta1, float beta2,
                                                          float eps, float wd, int64_t* step_dev, int32_t* scratch) {
    MMS_PDL_PROLOGUE();
    __shared__ AdamCoef s_c[MMS_MAX_ADAM_RANGES];
    const float lr = *lr_dev;
    for (int k = threadIdx.x; k < r.n; k += blockDim.x) s_c[k] = adam_coef(steps[r.slot[k]], lr, beta1, beta2);
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t base = 0;                       // virtual index of the range's first element
    for (int k = 0; k < r.n; ++k) {
        const AdamCoef c = s_c[k];
        int64_t j = (gt - base) % stride;
        if (j < 0) j += stride;
        for (; j < r.cnt[k]; j += stride) {
            adam_update(p, g, m, v, r.off[k] + j, c, beta1, beta2, eps, wd);
        }
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

int adam_ranges_from_host(const int64_t* table, int n, int64_t total, AdamRanges* r) {
    MMS_REQUIRE((table || n == 0) && n >= 0 && n <= MMS_MAX_ADAM_RANGES, "adam ranges: %d ranges, need 0..%d", n, MMS_MAX_ADAM_RANGES);
    r->n = n;
    for (int k = 0; k < n; ++k) {
        const int64_t off = table[3 * k], cnt = table[3 * k + 1], slot = table[3 * k + 2];
        MMS_REQUIRE(off >= 0 && cnt >= 1 && off + cnt <= total && slot >= 0 && slot <= INT32_MAX,
                    "adam ranges: range %d = (%lld, %lld, %lld) outside a buffer of %lld floats", k, (long long)off, (long long)cnt,
                    (long long)slot, (long long)total);
        for (int q = 0; q < k; ++q)
            MMS_REQUIRE(off + cnt <= r->off[q] || r->off[q] + r->cnt[q] <= off, "adam ranges: ranges %d and %d overlap", q, k);
        r->off[k] = off; r->cnt[k] = cnt; r->slot[k] = (int32_t)slot;
    }
    return MMS_OK;
}

int launch_head_fwd2(const float* src_a, int64_t lda, const float* src_b, int64_t ldb, int Hh, const float* w0, const float* b0,
                     const float* w3, const float* b3, int B, int H2, int nc, float p, uint64_t seed, uint64_t offset,
                     const int64_t* offset_dev, float* last_out, float* hid_out, float* logits, cudaStream_t st,
                     int64_t drop_row0) {
    MMS_REQUIRE(nc >= 1 && nc <= MAX_NC, "head: num_classes %d outside [1,%d]", nc, MAX_NC);
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(head_fwd_kernel, dim3(B), dim3(4 * HEAD_HID), H2 * sizeof(float), st, src_a, lda, src_b, ldb, Hh, w0, b0, w3, b3, H2, nc, p, seed, offset,
                                                             offset_dev, drop_row0, last_out, hid_out, logits);
    MMS_LAUNCH_CHECK("head_fwd_kernel");
    return MMS_OK;
}

int launch_head_ce_fused(const float* src_a, int64_t lda, const float* src_b, int64_t ldb, int Hh, const float* w0, const float* b0,
                         const float* w3, const float* b3, const int64_t* labels, int B, int H2, int nc, float p, uint64_t seed,
                         uint64_t offset, const int64_t* offset_dev, int div_batch, float* last_out, float* hid_out, float* logits,
                         float* dlogits, float* dhid, float* rowloss, int32_t* counter, float* loss_out, double* loss_sum_accum,
                         cudaStream_t st, const float* class_weight) {
    MMS_REQUIRE(nc >= 1 && nc <= MAX_NC, "head: num_classes %d outside [1,%d]", nc, MAX_NC);
    MMS_PROF_BEGIN(st);
    if (class_weight)
        MMS_LAUNCH(head_ce_fused_kernel<true>, dim3(B), dim3(4 * HEAD_HID), H2 * sizeof(float), st, src_a, lda, src_b, ldb, Hh, w0, b0, w3,
                   b3, labels, H2, nc, p, seed, offset, offset_dev, div_batch > 0 ? div_batch : B, last_out, hid_out, logits, dlogits,
                   dhid, rowloss, counter, loss_out, loss_sum_accum, class_weight);
    else
        MMS_LAUNCH(head_ce_fused_kernel<false>, dim3(B), dim3(4 * HEAD_HID), H2 * sizeof(float), st, src_a, lda, src_b, ldb, Hh, w0, b0, w3,
                   b3, labels, H2, nc, p, seed, offset, offset_dev, div_batch > 0 ? div_batch : B, last_out, hid_out, logits, dlogits,
                   dhid, rowloss, counter, loss_out, loss_sum_accum, nullptr);
    MMS_LAUNCH_CHECK("head_ce_fused_kernel");
    return MMS_OK;
}

int launch_head_fwd(const float* last, const float* w0, const float* b0, const float* w3, const float* b3, int B, int H2,
                    int nc, float p, uint64_t seed, uint64_t offset, const int64_t* offset_dev, float* hid_out, float* logits,
                    cudaStream_t st) {
    return launch_head_fwd2(last, H2, last + H2 / 2, H2, H2 / 2, w0, b0, w3, b3, B, H2, nc, p, seed, offset, offset_dev, nullptr,
                            hid_out, logits, st, 0);
}

int launch_head_bwd(const float* last, const float* hid, const float* dlogits, const float* w3, int B, int H2, int nc, float p,
                    uint64_t seed, uint64_t offset, const int64_t* offset_dev, float* dhid, float* dw0, float* db0, float* dw3,
                    float* db3, cudaStream_t st) {
    MMS_REQUIRE(nc >= 1 && nc <= MAX_NC, "head: num_classes %d outside [1,%d]", nc, MAX_NC);
    MMS_REQUIRE(B * sizeof(float) <= 40 * 1024, "head_bwd: batch %d too large for one CTA's shared memory", B);
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(head_bwd_kernel, dim3(HEAD_HID), dim3(128), B * sizeof(float), st, last, hid, dlogits, w3, B, H2, nc, p, seed, offset, offset_dev, dhid,
                                                              dw0, db0, dw3, db3);
    MMS_LAUNCH_CHECK("head_bwd_kernel");
    return MMS_OK;
}

int launch_cross_entropy(const float* logits, const int64_t* labels, int B, int nc, float* loss_out, float* dlogits,
                         double* loss_sum_accum, cudaStream_t st, int div_batch = 0, const float* class_weight = nullptr,
                         const double* norm = nullptr) {
    if (div_batch <= 0) div_batch = B;
    MMS_REQUIRE(nc >= 1 && nc <= MAX_NC, "cross_entropy: num_classes %d outside [1,%d]", nc, MAX_NC);
    MMS_REQUIRE(class_weight || !norm, "cross_entropy: a normaliser needs class weights");
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(cross_entropy_kernel, dim3(1), dim3(256), 0, st, logits, labels, B, nc, loss_out, dlogits, loss_sum_accum, div_batch,
               class_weight, norm);
    MMS_LAUNCH_CHECK("cross_entropy_kernel");
    return MMS_OK;
}

// out[0] = sum_b w[y_b] over the labels in [0, nc), float64, one warp in a fixed order: the local normaliser of the weighted
// cross entropy, written into a slot the data-parallel exchange sums over the ranks.
__global__ void __launch_bounds__(32) class_weight_sum_kernel(const int64_t* __restrict__ labels, int B, int nc,
                                                              const float* __restrict__ class_weight, double* __restrict__ out) {
    MMS_PDL_PROLOGUE();
    double ws = 0.0;
    for (int b = threadIdx.x; b < B; b += 32) {
        const int64_t y = labels[b];
        if (y >= 0 && y < nc) ws += (double)class_weight[y];
    }
    ws = warp_sum(ws);
    if (threadIdx.x == 0) out[0] = ws;
}

int launch_class_weight_sum(const int64_t* labels, int B, int nc, const float* class_weight, double* out, cudaStream_t st) {
    MMS_REQUIRE(nc >= 1 && nc <= MAX_NC, "class_weight_sum: num_classes %d outside [1,%d]", nc, MAX_NC);
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(class_weight_sum_kernel, dim3(1), dim3(32), 0, st, labels, B, nc, class_weight, out);
    MMS_LAUNCH_CHECK("class_weight_sum_kernel");
    return MMS_OK;
}

int launch_adam(float* p, const float* g, float* m, float* v, int64_t n, const float* lr_dev, float beta1, float beta2,
                float eps, float wd, int64_t* step_dev, int32_t* scratch, cudaStream_t st) {
    const int blocks = (int)((n + 255) / 256 < 592 ? (n + 255) / 256 : 592);
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(adam_flat_kernel, dim3(blocks > 0 ? blocks : 1), dim3(256), 0, st, p, g, m, v, n, lr_dev, beta1, beta2, eps, wd, step_dev, scratch);
    MMS_LAUNCH_CHECK("adam_flat_kernel");
    return MMS_OK;
}

int launch_adam_ranges(float* p, const float* g, float* m, float* v, const AdamRanges& r, int64_t* steps, const float* lr_dev,
                       float beta1, float beta2, float eps, float wd, int64_t* step_dev, int32_t* scratch, cudaStream_t st) {
    int64_t n = 0;
    for (int k = 0; k < r.n; ++k) n += r.cnt[k];
    const int blocks = (int)((n + 255) / 256 < 592 ? (n + 255) / 256 : 592);
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(adam_ranges_kernel, dim3(blocks > 0 ? blocks : 1), dim3(256), 0, st, p, g, m, v, r, steps, lr_dev, beta1, beta2, eps, wd,
               step_dev, scratch);
    MMS_LAUNCH_CHECK("adam_ranges_kernel");
    return MMS_OK;
}

}  // namespace mms

using namespace mms;

extern "C" int mms_head_fwd(const float* last, const float* w0, const float* b0, const float* w3, const float* b3, int32_t B,
                            int32_t H2, int32_t nc, float dropout_p, uint64_t rng_seed, uint64_t rng_offset,
                            const int64_t* rng_offset_dev, float* hid_out, float* logits, mms_stream_t stream) {
    MMS_REQUIRE(last && w0 && b0 && w3 && b3 && hid_out && logits && B > 0, "head_fwd: bad arguments");
    return launch_head_fwd(last, w0, b0, w3, b3, B, H2, nc, dropout_p, rng_seed, rng_offset, rng_offset_dev, hid_out, logits,
                           (cudaStream_t)stream);
}
extern "C" int mms_head_bwd(const float* last, const float* hid, const float* dlogits, const float* w3, int32_t B, int32_t H2,
                            int32_t nc, float dropout_p, uint64_t rng_seed, uint64_t rng_offset, const int64_t* rng_offset_dev,
                            float* dhid, float* dw0, float* db0, float* dw3, float* db3, mms_stream_t stream) {
    MMS_REQUIRE(last && hid && dlogits && w3 && dw0 && db0 && dw3 && db3 && B > 0, "head_bwd: bad arguments");
    return launch_head_bwd(last, hid, dlogits, w3, B, H2, nc, dropout_p, rng_seed, rng_offset, rng_offset_dev, dhid, dw0, db0, dw3,
                           db3, (cudaStream_t)stream);
}
extern "C" int mms_cross_entropy(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes, float* loss_out,
                                 float* dlogits, double* loss_sum_accum, mms_stream_t stream) {
    MMS_REQUIRE(logits && labels && loss_out && batch > 0, "cross_entropy: bad arguments");
    return launch_cross_entropy(logits, labels, batch, num_classes, loss_out, dlogits, loss_sum_accum, (cudaStream_t)stream, batch);
}
extern "C" int mms_cross_entropy_partial(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes,
                                         int32_t global_batch, float* loss_out, float* dlogits, double* loss_sum_accum,
                                         mms_stream_t stream) {
    MMS_REQUIRE(logits && labels && loss_out && batch > 0 && global_batch >= batch, "cross_entropy_partial: bad arguments");
    return launch_cross_entropy(logits, labels, batch, num_classes, loss_out, dlogits, loss_sum_accum, (cudaStream_t)stream, global_batch);
}
extern "C" int mms_cross_entropy_weighted(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes,
                                          const float* class_weight, const double* norm_dev, float* loss_out, float* dlogits,
                                          double* loss_sum_accum, mms_stream_t stream) {
    MMS_REQUIRE(logits && labels && loss_out && batch > 0, "cross_entropy_weighted: bad arguments");
    return launch_cross_entropy(logits, labels, batch, num_classes, loss_out, dlogits, loss_sum_accum, (cudaStream_t)stream, batch,
                                class_weight, norm_dev);
}
extern "C" int mms_class_weight_sum(const int64_t* labels, int32_t batch, int32_t num_classes, const float* class_weight,
                                    double* out, mms_stream_t stream) {
    MMS_REQUIRE(labels && class_weight && out && batch > 0, "class_weight_sum: bad arguments");
    return launch_class_weight_sum(labels, batch, num_classes, class_weight, out, (cudaStream_t)stream);
}
extern "C" int mms_adam_flat_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                                  const float* lr_dev, float beta1, float beta2, float eps, float weight_decay, int64_t* step_dev,
                                  int32_t* scratch_dev, mms_stream_t stream) {
    MMS_REQUIRE(params && grads && exp_avg && exp_avg_sq && lr_dev && step_dev && scratch_dev && n > 0, "adam_flat_step: bad arguments");
    return launch_adam(params, grads, exp_avg, exp_avg_sq, n, lr_dev, beta1, beta2, eps, weight_decay, step_dev, scratch_dev,
                       (cudaStream_t)stream);
}
extern "C" int mms_adam_ranges_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, const int64_t* ranges_host,
                                    int32_t nranges, int64_t* steps_dev, const float* lr_dev, float beta1, float beta2, float eps,
                                    float weight_decay, int64_t* step_dev, int32_t* scratch_dev, mms_stream_t stream) {
    MMS_REQUIRE(params && grads && exp_avg && exp_avg_sq && steps_dev && lr_dev && step_dev && scratch_dev, "adam_ranges_step: bad arguments");
    AdamRanges r;
    const int rc = adam_ranges_from_host(ranges_host, nranges, INT64_MAX / 2, &r);
    if (rc) return rc;
    return launch_adam_ranges(params, grads, exp_avg, exp_avg_sq, r, steps_dev, lr_dev, beta1, beta2, eps, weight_decay, step_dev,
                              scratch_dev, (cudaStream_t)stream);
}
