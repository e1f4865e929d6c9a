// Backward pass of the CNN encoder (reverse of reference models.py:45-53 and 24-31), the default path of a training step
// when the shapes allow it (T % 64 == 0, cnn_out_channels == 32, no input gradient requested):
//
//   pool_bwd_tm_kernel    MaxPool1d(3,2,1) + ReLU backward of stage 2 and the two BatchNorm reductions (sum dyn, sum dyn*xhat).
//                         The upstream gradient is time-major [B, L, C] (the GRU's layout): a thread owns ONE channel
//                         (lanes run over channels, so those rows are read as full 128-byte lines) and 8 consecutive
//                         positions (two 128-bit loads / stores in the channel-major tensors, every 32-byte sector used in full).
//   conv2_bwd_kernel      BatchNorm-backward apply + BOTH gradients of Conv1d(16,32,k5,s2,p2) from one staged tile: warps 0-1
//                         the input gradient (8 position pairs x 4 input channels per thread), warps 2-3 the weight
//                         gradient (8 output x 2 input channels x 5 taps per thread, two positions per iteration).  Partial
//                         weight gradients leave through a scratch buffer (one coalesced 10 KB store per CTA, no atomics)
//                         and are summed by wgrad_reduce_kernel on a side stream.
//   pool_bwd_ncl_kernel   the same pool / ReLU backward for stage 1 (channel-major upstream gradient): pure streaming, 8
//                         elements per thread, every load of a thread issued before the first use.
//   conv1_bwd_kernel      G[b,o,c,k] = sum_l dy1[b,o,l] * x[b,c,2l+k-3] per batch row, from which BOTH remaining gradients of
//                         stage 1 follow:  dW1[o,c,k] += gate[b,c] * G  and  dgate[b,c] = sum_{o,k} W1[o,c,k] * G  (the input
//                         gradient of conv1 is never formed: it was only ever reduced against x), then the ChannelAttention
//                         parameter gradients of the row.  A warp owns an input channel, lanes run over positions with all
//                         16 x 7 partial sums in registers (56 packed FFMA2 per position against 16 + 8 shared-memory words).
//                         The chunks of a row meet through a scratch buffer; the LAST CTA of a row (a counter) finishes it.
//
// What the first versions of these kernels (and their predecessors in conv_bn_pool.cu) lost their time on -- ncu, round 2:
// 40-80 % of the stall samples sat on tile STAGING (a loop of "load, use" fetches one L2 latency per iteration), the rest on
// barriers; the FMA pipes were 2-5 % busy.  So every tile here arrives by bulk asynchronous copies (cp.async.bulk, one
// instruction per row, completion on an mbarrier: all rows of a tile in flight at once), rows outside the tensor are zero
// filled by the issuing lane, and a CTA has exactly one block barrier between staging and compute.
#include "conv_common.cuh"
#include "tc_common.cuh"

namespace mms {

// Columns [g0, g0 + n) of a row of `len` floats -> dst[0, n): the part inside the row by ONE bulk copy, the rest zeros (plain
// stores of the calling lane).  g0, n, len multiples of 4 and both pointers 16-byte aligned.  Arrives once on `bar`.
__device__ __forceinline__ void row_load(float* dst, const float* row, int g0, int n, int len, uint64_t* bar) {
    const int lo = g0 > 0 ? g0 : 0, hi = g0 + n < len ? g0 + n : len;
    if (hi > lo) {
        mbar_expect_tx(bar, (uint32_t)(hi - lo) * 4u);
        bulk_g2s(dst + (lo - g0), row + lo, (uint32_t)(hi - lo) * 4u, bar);
        for (int i = 0; i < lo - g0; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int i = hi - g0; i < n; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
        mbar_arrive(bar);
        for (int i = 0; i < n; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

__device__ __forceinline__ float2 bc2(float v) { return make_float2(v, v); }

// ------------------------------------------------------------------------------------------------------------------
// Pool / ReLU backward of one element given z = relu(bn(y)) at i-2 .. i+2 and the upstream gradients of the windows around
// it.  Window j covers (2j-1, 2j, 2j+1); the FIRST maximal element wins (ATen: val > maxval), -inf padding never wins.
//   even i: only window j = i/2 (i is its centre);  odd i: windows ja = (i+1)/2 (i is its first element) and jb = (i-1)/2 (last)
__device__ __forceinline__ float pool_bwd_even(float zm1, float z0, float zp1, float dj) {
    return (!(zm1 >= z0) && !(zp1 > z0)) ? dj : 0.f;
}
__device__ __forceinline__ float pool_bwd_odd(float zm2, float zm1, float z0, float zp1, float zp2, float dja, float djb) {
    float d = 0.f;
    if (!(zp1 > z0) && !(zp2 > z0)) d += dja;
    if (!(zm2 >= z0) && !(zm1 >= z0)) d += djb;
    return d;
}

// 8 consecutive elements i0 .. i0+7 (i0 % 8 == 0) of one (b, c) row: y4[0..3] = y[i0-4 .. i0+11] (16 values), dj[0..4] =
// upstream gradient of the windows i0/2 .. i0/2+4 (0 where the window does not exist).  Returns dyn[8] and adds to s1 / s2.
__device__ __forceinline__ void pool_bwd_8(const float (&yv)[16], const float (&dj)[5], int i0, int Lin, float a, float bsh,
                                           float mean, float inv, float (&dyn)[8], float& s1, float& s2) {
    float z[12];      // z[t] = relu(bn(y[i0 - 2 + t])), -inf outside the row
#pragma unroll
    for (int t = 0; t < 12; ++t) {
        const int i = i0 - 2 + t;
        z[t] = (i >= 0 && i < Lin) ? fmaxf(fmaf(a, yv[t + 2], bsh), 0.f) : -INFINITY;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const float z0 = z[e + 2];
        float d;
        if ((e & 1) == 0) d = pool_bwd_even(z[e + 1], z0, z[e + 3], dj[e >> 1]);
        else d = pool_bwd_odd(z[e], z[e + 1], z0, z[e + 3], z[e + 4], dj[(e + 1) >> 1], dj[(e - 1) >> 1]);
        d = (z0 > 0.f && i0 + e < Lin) ? d : 0.f;
        dyn[e] = d;
        s1 += d;
        s2 = fmaf(d, (yv[e + 4] - mean) * inv, s2);
    }
}

// ---- stage 2: time-major upstream gradient --------------------------------------------------------------------------
// grid = (ceil(Lin / (8 * NS * PB_ITERS)), B), block = 256 = C channels x NS position slots; a thread handles PB_ITERS groups
// of 8 positions (2 or 4: MMS_POOL_TM_ITERS).  Lin % 8 == 0.
template <int C, int PB_ITERS>
__global__ void __launch_bounds__(256) pool_bwd_tm_kernel(const float* __restrict__ y, const double* __restrict__ stats,
                                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                                          const float* __restrict__ rm, const float* __restrict__ rv,
                                                          const float* __restrict__ dout, int Bn, int Lin, int Lout, int training,
                                                          float* __restrict__ dy, double* __restrict__ red) {
    MMS_PDL_PROLOGUE();
    constexpr int NS = 256 / C;
    __shared__ float s_part[2][NS][C];
    const int tid = threadIdx.x, c = tid % C, slot = tid / C;
    const int b = blockIdx.y;
    const float* row = y + ((size_t)b * C + c) * Lin;
    float* dyrow = dy + ((size_t)b * C + c) * Lin;
    const float* dcol = dout + (size_t)b * Lout * C + c;
    float yv[PB_ITERS][16], dj[PB_ITERS][5];
    int i0s[PB_ITERS];
#pragma unroll
    for (int it = 0; it < PB_ITERS; ++it) {
        const int i0 = ((blockIdx.x * PB_ITERS + it) * NS + slot) * 8;
        i0s[it] = i0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int i = i0 - 4 + 4 * q;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i >= 0 && i < Lin) v = __ldg(reinterpret_cast<const float4*>(row + i));
            yv[it][4 * q] = v.x; yv[it][4 * q + 1] = v.y; yv[it][4 * q + 2] = v.z; yv[it][4 * q + 3] = v.w;
        }
#pragma unroll
        for (int t = 0; t < 5; ++t) {
            const int j = (i0 >> 1) + t;
            dj[it][t] = (i0 < Lin && j < Lout) ? __ldg(dcol + (size_t)j * C) : 0.f;
        }
    }
    const BnAffine af = bn_affine(training, stats, gamma, beta, rm, rv, c, C, (double)Bn * (double)Lin);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int it = 0; it < PB_ITERS; ++it) {
        const int i0 = i0s[it];
        if (i0 < Lin) {
            float dyn[8];
            pool_bwd_8(yv[it], dj[it], i0, Lin, af.a, af.b, af.mean, af.inv, dyn, s1, s2);
            *reinterpret_cast<float4*>(dyrow + i0) = make_float4(dyn[0], dyn[1], dyn[2], dyn[3]);
            *reinterpret_cast<float4*>(dyrow + i0 + 4) = make_float4(dyn[4], dyn[5], dyn[6], dyn[7]);
        }
    }
    s_part[0][slot][c] = s1;
    s_part[1][slot][c] = s2;
    __syncthreads();
    if (tid < 2 * C) {
        const int which = tid / C, cc = tid % C;
        float t = 0.f;
#pragma unroll
        for (int s = 0; s < NS; ++s) t += s_part[which][s][cc];
        atomicAdd(red + which * C + cc, (double)t);      // red[0][c] = sum dyn, red[1][c] = sum dyn * xhat
    }
}

// ---- stage 1: channel-major upstream gradient -----------------------------------------------------------------------
// grid = (ceil(Lin / 2048), C, B), block = 256: 8 consecutive elements per thread.  Lin % 8 == 0, Lout % 4 == 0.
__global__ void __launch_bounds__(256) pool_bwd_ncl_kernel(const float* __restrict__ y, const double* __restrict__ stats,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                           const float* __restrict__ rm, const float* __restrict__ rv,
                                                           const float* __restrict__ dout, int Bn, int C, int Lin, int Lout,
                                                           int training, float* __restrict__ dy, double* __restrict__ red) {
    MMS_PDL_PROLOGUE();
    __shared__ float s_part[2][8];
    const int tid = threadIdx.x, c = blockIdx.y, b = blockIdx.z;
    const int i0 = (blockIdx.x * 256 + tid) * 8;
    const float* row = y + ((size_t)b * C + c) * Lin;
    const float* drow = dout + ((size_t)b * C + c) * Lout;
    float yv[16], dj[5];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int i = i0 - 4 + 4 * q;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i >= 0 && i < Lin) v = __ldg(reinterpret_cast<const float4*>(row + i));
        yv[4 * q] = v.x; yv[4 * q + 1] = v.y; yv[4 * q + 2] = v.z; yv[4 * q + 3] = v.w;
    }
    {
        const int j0 = i0 >> 1;      // multiple of 4
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i0 < Lin && j0 < Lout) v = __ldg(reinterpret_cast<const float4*>(drow + j0));
        dj[0] = v.x; dj[1] = v.y; dj[2] = v.z; dj[3] = v.w;
        dj[4] = (i0 < Lin && j0 + 4 < Lout) ? __ldg(drow + j0 + 4) : 0.f;
    }
    const BnAffine af = bn_affine(training, stats, gamma, beta, rm, rv, c, C, (double)Bn * (double)Lin);
    float s1 = 0.f, s2 = 0.f;
    if (i0 < Lin) {
        float dyn[8];
        pool_bwd_8(yv, dj, i0, Lin, af.a, af.b, af.mean, af.inv, dyn, s1, s2);
        float* dyrow = dy + ((size_t)b * C + c) * Lin;
        *reinterpret_cast<float4*>(dyrow + i0) = make_float4(dyn[0], dyn[1], dyn[2], dyn[3]);
        *reinterpret_cast<float4*>(dyrow + i0 + 4) = make_float4(dyn[4], dyn[5], dyn[6], dyn[7]);
    }
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if ((tid & 31) == 0) { s_part[0][tid >> 5] = s1; s_part[1][tid >> 5] = s2; }
    __syncthreads();
    if (tid < 2) {
        float t = 0.f;
#pragma unroll
        for (int wq = 0; wq < 8; ++wq) t += s_part[tid][wq];
        atomicAdd(red + tid * C + c, (double)t);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// conv2_bwd_kernel.  grid = (ceil(Lout / 128), B), block = 128.  Tile: conv2 output positions m in [m0, m0 + 128).
//   raw_d / raw_y [32][136]   un-normalised gradient and conv2 output, m in [m0 - 4, m0 + 132)   (bulk copies, 16-byte aligned)
//   p1s [2][16][140]          pooled stage-1 activations for the two weight-gradient warps: j in [2 m0 + 128 h - 4, ... + 140)
//   wd [32 * 5][16]           wd[(o*5 + k)*16 + ci] = w[o][ci][k]
//   dys [32][132]             dy2[o][m0 - 1 + mm]  (BatchNorm backward applied; 0 outside the tensor)   -> input gradient
//   dyT [130][36]             the same values, position-major                                          -> weight gradient
constexpr int C2B_TM = 128, C2B_RW = 136, C2B_PW = 140, C2B_DS = 132, C2B_CO = 32, C2B_TS = C2B_CO + 4, C2B_NW = C2B_CO * 80;
constexpr int C2B_SMEM_FLOATS = 2 * C2B_CO * C2B_RW + 2 * 16 * C2B_PW + C2B_NW + C2B_CO * C2B_DS + 130 * C2B_TS;

// DGRAD = false: the weight gradient alone (stage 1 needs no gradient, frozen segments): warps 0-1 stop after the staging.
template <bool DGRAD>
__device__ __forceinline__ void conv2_bwd_body(const float* __restrict__ dyn, const float* __restrict__ wdg,
                                               const float* __restrict__ p1, float* __restrict__ dp1,
                                               float* __restrict__ dw_part, int Lin, int Lout, const BnBwd bn) {
    MMS_PDL_TRIGGER();
    constexpr int CO2 = C2B_CO;
    extern __shared__ __align__(128) float c2b_smem[];
    float* raw_d = c2b_smem;
    float* raw_y = raw_d + CO2 * C2B_RW;
    float* p1s = raw_y + CO2 * C2B_RW;
    float* wd = p1s + 2 * 16 * C2B_PW;
    float* dys = wd + C2B_NW;
    float* dyT = dys + CO2 * C2B_DS;
    __shared__ __align__(8) uint64_t bar;
    __shared__ float s_bn[CO2][5];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y, m0 = blockIdx.x * C2B_TM;
    const bool fold = bn.y != nullptr;
    if (tid == 0) {
        mbar_init(&bar, (uint32_t)(CO2 * (fold ? 2 : 1) + 32 + 1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    MMS_PDL_WAIT();
    __syncthreads();
    if (warp == 0) {
        {
            const int r = lane;       // CO2 == 32: one row of each tile per lane
            row_load(raw_d + r * C2B_RW, dyn + ((size_t)b * CO2 + r) * Lout, m0 - 4, C2B_RW, Lout, &bar);
            if (fold) row_load(raw_y + r * C2B_RW, bn.y + ((size_t)b * CO2 + r) * Lout, m0 - 4, C2B_RW, Lout, &bar);
        }
        const int h = lane >> 4, ci = lane & 15;
        row_load(p1s + (h * 16 + ci) * C2B_PW, p1 + ((size_t)b * 16 + ci) * Lin, 2 * m0 + 128 * h - 4, C2B_PW, Lin, &bar);
        if (lane == 0) {              // the weights, already in the [o][k][ci] order the input gradient reads (conv2_w_relayout_kernel)
            mbar_expect_tx(&bar, (uint32_t)C2B_NW * 4u);
            bulk_g2s(wd, wdg, (uint32_t)C2B_NW * 4u, &bar);
        }
    } else if (warp == 1 && fold) {   // constants of the folded BatchNorm backward (float64 arithmetic) beside the copies
        const int o = lane;
        const double n = (double)bn.Bstat * (double)Lout;
        const BnAffine af = bn_affine(bn.training, bn.stats, bn.gamma, bn.beta, bn.rm, bn.rv, o, CO2, n);
        s_bn[o][0] = af.a;
        s_bn[o][1] = af.mean;
        s_bn[o][2] = af.inv;
        s_bn[o][3] = bn.training ? (float)(bn.red[o] / n) : 0.f;
        s_bn[o][4] = bn.training ? (float)(bn.red[CO2 + o] / n) : 0.f;
        if (blockIdx.x == 0 && blockIdx.y == 0) {      // dgamma / dbeta once per launch
            if (bn.dgamma) bn.dgamma[o] += bn.grad_scale * (float)bn.red[CO2 + o];
            if (bn.dbeta) bn.dbeta[o] += bn.grad_scale * (float)bn.red[o];
        }
    }
    mbar_wait(&bar, 0);
    __syncthreads();
    {   // dyn -> dy2 (BnBwd) into both layouts, zero outside the tensor: 4 threads per output channel, positions q, q + 4, ...
        const int o = tid >> 2, q = tid & 3;
        float ca = 1.f, cm1 = 0.f, cmean = 0.f, cim2 = 0.f;
        if (fold) { ca = s_bn[o][0]; cm1 = s_bn[o][3]; cmean = s_bn[o][1]; cim2 = s_bn[o][2] * s_bn[o][4]; }
        const float* rd = raw_d + o * C2B_RW + 3;
        const float* ry = raw_y + o * C2B_RW + 3;
#pragma unroll 4
        for (int mm = q; mm < 130; mm += 4) {
            const int m = m0 - 1 + mm;
            float v = 0.f;
            if (m >= 0 && m < Lout) {
                v = rd[mm];
                if (fold) v = ca * (v - cm1 - (ry[mm] - cmean) * cim2);
            }
            dys[o * C2B_DS + mm] = v;
            dyT[mm * C2B_TS + o] = v;
        }
    }
    __syncthreads();

    if (warp < 2) {
        if (!DGRAD) return;
        // ===== input gradient: pairs u = m0 + 64 warp + 8 pg + e (positions 2u, 2u + 1), input channels 4 cg .. 4 cg + 3 =====
        //   even j = 2u   : taps k = 0, 2, 4 with m = u + 1, u, u - 1;    odd j = 2u + 1 : taps k = 1, 3 with m = u + 1, u
        const int pg = (lane & 3) | ((lane >> 2) & 4), cg = (lane >> 2) & 3;     // a quarter-warp = 4 pair groups x 2 channel groups
        float2 ae[8][2], ao[8][2];
#pragma unroll
        for (int e = 0; e < 8; ++e)
#pragma unroll
            for (int i = 0; i < 2; ++i) { ae[e][i] = make_float2(0.f, 0.f); ao[e][i] = make_float2(0.f, 0.f); }
        const float* drow = dys + 64 * warp + 8 * pg;
        const float* wrow = wd + 4 * cg;
#pragma unroll 2
        for (int o = 0; o < CO2; ++o) {
            float d[10];
            {
                const float4 v0 = *reinterpret_cast<const float4*>(drow + o * C2B_DS);
                const float4 v1 = *reinterpret_cast<const float4*>(drow + o * C2B_DS + 4);
                const float2 v2 = *reinterpret_cast<const float2*>(drow + o * C2B_DS + 8);
                d[0] = v0.x; d[1] = v0.y; d[2] = v0.z; d[3] = v0.w; d[4] = v1.x; d[5] = v1.y; d[6] = v1.z; d[7] = v1.w;
                d[8] = v2.x; d[9] = v2.y;
            }
            float2 wk[5][2];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const float4 t = *reinterpret_cast<const float4*>(wrow + (o * 5 + k) * 16);
                wk[k][0] = make_float2(t.x, t.y);
                wk[k][1] = make_float2(t.z, t.w);
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float2 dm = bc2(d[e]), dc = bc2(d[e + 1]), dp = bc2(d[e + 2]);       // dy[u - 1], dy[u], dy[u + 1]
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    ae[e][i] = __ffma2_rn(wk[0][i], dp, ae[e][i]);
                    ae[e][i] = __ffma2_rn(wk[2][i], dc, ae[e][i]);
                    ae[e][i] = __ffma2_rn(wk[4][i], dm, ae[e][i]);
                    ao[e][i] = __ffma2_rn(wk[1][i], dp, ao[e][i]);
                    ao[e][i] = __ffma2_rn(wk[3][i], dc, ao[e][i]);
                }
            }
        }
        const int j0 = 2 * (m0 + 64 * warp + 8 * pg);          // 16 consecutive positions per thread and channel
#pragma unroll
        for (int i = 0; i < 2; ++i) {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                float* dst = dp1 + ((size_t)b * 16 + 4 * cg + 2 * i + hh) * Lin + j0;
                float v[16];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    v[2 * e] = hh ? ae[e][i].y : ae[e][i].x;
                    v[2 * e + 1] = hh ? ao[e][i].y : ao[e][i].x;
                }
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (j0 + 4 * q < Lin) *reinterpret_cast<float4*>(dst + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            }
        }
    } else {
        // ===== weight gradient: dW[o][ci][k] = sum_m dy2[o][m] * p1[ci][2m + k - 2], m in [m0 + 64 h, m0 + 64 h + 64) =====
        // thread: output channels 8 og .. 8 og + 7 (packed in pairs), input channels 2 cg2, 2 cg2 + 1, all 5 taps
        const int h = warp - 2, og = lane & 3, cg2 = lane >> 2;
        float2 acc[4][2][5];
#pragma unroll
        for (int op = 0; op < 4; ++op)
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
                for (int k = 0; k < 5; ++k) acc[op][c][k] = make_float2(0.f, 0.f);
        const float* dT = dyT + (64 * h + 1) * C2B_TS + 8 * og;            // row mm = 64 h + mi + 1
        const float* xr = p1s + (h * 16 + 2 * cg2) * C2B_PW + 2;           // tile column of tap k at position mi: 2 mi + k + 2
#pragma unroll 2
        for (int mi = 0; mi < 64; mi += 2) {
            float2 dy2[2][4];
#pragma unroll
            for (int mq = 0; mq < 2; ++mq) {
                const float4 a0 = *reinterpret_cast<const float4*>(dT + (mi + mq) * C2B_TS);
                const float4 a1 = *reinterpret_cast<const float4*>(dT + (mi + mq) * C2B_TS + 4);
                dy2[mq][0] = make_float2(a0.x, a0.y); dy2[mq][1] = make_float2(a0.z, a0.w);
                dy2[mq][2] = make_float2(a1.x, a1.y); dy2[mq][3] = make_float2(a1.z, a1.w);
            }
            float xw[2][8];
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float2 t = *reinterpret_cast<const float2*>(xr + c * C2B_PW + 2 * mi + 2 * q);
                    xw[c][2 * q] = t.x; xw[c][2 * q + 1] = t.y;
                }
#pragma unroll
            for (int mq = 0; mq < 2; ++mq)
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        const float2 xv = bc2(xw[c][k + 2 * mq]);
#pragma unroll
                        for (int op = 0; op < 4; ++op) acc[op][c][k] = __ffma2_rn(dy2[mq][op], xv, acc[op][c][k]);
                    }
        }
        // the two warps' partial sums meet in shared memory (raw_d is dead), then one coalesced store of the CTA's 32*16*5 values
        float* ex = raw_d;
        if (h == 1) {
#pragma unroll
            for (int op = 0; op < 4; ++op)
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        ex[((8 * og + 2 * op) * 16 + 2 * cg2 + c) * 5 + k] = acc[op][c][k].x;
                        ex[((8 * og + 2 * op + 1) * 16 + 2 * cg2 + c) * 5 + k] = acc[op][c][k].y;
                    }
        }
        asm volatile("bar.sync 1, 64;" ::: "memory");
        if (h == 0) {
#pragma unroll
            for (int op = 0; op < 4; ++op)
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        ex[((8 * og + 2 * op) * 16 + 2 * cg2 + c) * 5 + k] += acc[op][c][k].x;
                        ex[((8 * og + 2 * op + 1) * 16 + 2 * cg2 + c) * 5 + k] += acc[op][c][k].y;
                    }
        }
        asm volatile("bar.sync 1, 64;" ::: "memory");
        float4* dstp = reinterpret_cast<float4*>(dw_part + ((size_t)b * gridDim.x + blockIdx.x) * C2B_NW);
        const float4* srcp = reinterpret_cast<const float4*>(ex);
        for (int i = tid - 64; i < C2B_NW / 4; i += 64) dstp[i] = srcp[i];
    }
}

__global__ void __launch_bounds__(128) conv2_bwd_kernel(const float* __restrict__ dyn, const float* __restrict__ wdg,
                                                        const float* __restrict__ p1, float* __restrict__ dp1,
                                                        float* __restrict__ dw_part, int Lin, int Lout, const BnBwd bn) {
    conv2_bwd_body<true>(dyn, wdg, p1, dp1, dw_part, Lin, Lout, bn);
}

__global__ void __launch_bounds__(128) conv2_wgrad_bwd_kernel(const float* __restrict__ dyn, const float* __restrict__ wdg,
                                                              const float* __restrict__ p1, float* __restrict__ dw_part, int Lin,
                                                              int Lout, const BnBwd bn) {
    conv2_bwd_body<false>(dyn, wdg, p1, nullptr, dw_part, Lin, Lout, bn);
}

// wd[(o*5 + k)*16 + ci] = w[o][ci][k]: the order conv2_bwd_kernel's input-gradient warps read (one bulk copy per CTA instead of a
// strided gather by every CTA); runs on a side stream at the start of the backward pass.
__global__ void __launch_bounds__(256) conv2_w_relayout_kernel(const float* __restrict__ w, int n, float* __restrict__ wd) {
    const int idx = blockIdx.x * 256 + threadIdx.x;
    if (idx >= n) return;
    const int o = idx / 80, r = idx - o * 80, ci = r / 5, k = r - ci * 5;
    wd[(o * 5 + k) * 16 + ci] = __ldg(w + idx);
}

// dw[idx] += sum_p part[p][idx].  grid = (ceil(n / 256), S), block = 256: block (x, s) sums the partials s, s + S, ...
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ part, int P, int n, float* __restrict__ dw) {
    const int idx = blockIdx.x * 256 + threadIdx.x;
    if (idx >= n) return;
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    const int S = gridDim.y;
    for (int p = blockIdx.y; p < P; p += 4 * S) {
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (p + u * S < P) s[u] += __ldg(part + (size_t)(p + u * S) * n + idx);
    }
    atomicAdd(dw + idx, (s[0] + s[1]) + (s[2] + s[3]));
}

// ------------------------------------------------------------------------------------------------------------------
// conv1_bwd_kernel.  grid = (NCH, B), block = 32 * NW.  CTA (chunk, b) owns the conv1 output positions [chunk * CH, + CH) of
// batch row b (CH % 32 == 0).  dynamic smem: xs [C][2 CH + 8] (x columns [2 l0 - 4, 2 l0 + 2 CH + 4)) | dys [16][CH] | ys [16][CH]
// | s_G [C * 112].  gp: scratch [B][NCH][C * 112]; counter: [B] zeroed before the launch.
__global__ void __launch_bounds__(256) conv1_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dyn,
                                                        const float* __restrict__ w, const float* __restrict__ gate,
                                                        const float* __restrict__ mean, const float* __restrict__ ca_w1,
                                                        const float* __restrict__ ca_w2, int C, int A, int T, int Lout, int CH,
                                                        float* __restrict__ gp, int* __restrict__ counter, float* __restrict__ dw,
                                                        float* __restrict__ dca_w1, float* __restrict__ dca_w2, const BnBwd bn) {
    MMS_PDL_TRIGGER();
    extern __shared__ __align__(128) float c1b_smem[];
    const int XS = 2 * CH + 8;
    float* xs = c1b_smem;
    float* dys = xs + C * XS;
    float* ys = dys + 16 * CH;
    float* s_G = ys + 16 * CH;
    __shared__ __align__(8) uint64_t bar;
    __shared__ float s_bn[16][5];
    __shared__ float s_dgr[16], s_dg[16], s_hid[4], s_dh[4];
    __shared__ int s_last;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, NT = blockDim.x, NW = NT >> 5;
    const int b = blockIdx.y, chunk = blockIdx.x, NCH = gridDim.x;
    const int l0 = chunk * CH;
    const bool fold = bn.y != nullptr;
    if (tid == 0) {
        mbar_init(&bar, (uint32_t)(C + (fold ? 32 : 16)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    MMS_PDL_WAIT();
    __syncthreads();
    if (warp == 0) {
        if (lane < C) row_load(xs + lane * XS, x + ((size_t)b * C + lane) * T, 2 * l0 - 4, XS, T, &bar);
        if (lane < 16) row_load(dys + lane * CH, dyn + ((size_t)b * 16 + lane) * Lout, l0, CH, Lout, &bar);
        else if (fold) row_load(ys + (lane - 16) * CH, bn.y + ((size_t)b * 16 + lane - 16) * Lout, l0, CH, Lout, &bar);
    }
    // constants of the folded BatchNorm backward: the second warp beside the copies (the only warp of a one-channel model after them)
    if (warp == (NW > 1 ? 1 : 0) && fold && lane < 16) {
        const int o = lane;
        const double n = (double)bn.Bstat * (double)Lout;
        const BnAffine af = bn_affine(bn.training, bn.stats, bn.gamma, bn.beta, bn.rm, bn.rv, o, 16, n);
        s_bn[o][0] = af.a;
        s_bn[o][1] = af.mean;
        s_bn[o][2] = af.inv;
        s_bn[o][3] = bn.training ? (float)(bn.red[o] / n) : 0.f;
        s_bn[o][4] = bn.training ? (float)(bn.red[16 + o] / n) : 0.f;
        if (chunk == 0 && b == 0) {                       // dgamma / dbeta once per launch
            if (bn.dgamma) bn.dgamma[o] += bn.grad_scale * (float)bn.red[16 + o];
            if (bn.dbeta) bn.dbeta[o] += bn.grad_scale * (float)bn.red[o];
        }
    }
    mbar_wait(&bar, 0);
    __syncthreads();
    if (fold) {         // dyn -> dy1 in place (rows beyond the tensor stay zero): a warp per output channel, 128-bit accesses
        const int nl = Lout - l0 < CH ? Lout - l0 : CH;
        for (int o = warp; o < 16; o += NW) {
            const float ca = s_bn[o][0], cm1 = s_bn[o][3], cmean = s_bn[o][1], cim2 = s_bn[o][2] * s_bn[o][4];
            float4* dr = reinterpret_cast<float4*>(dys + o * CH);
            const float4* yr = reinterpret_cast<const float4*>(ys + o * CH);
            for (int q = lane; 4 * q < nl; q += 32) {
                float4 d = dr[q];
                const float4 yv = yr[q];
                d.x = ca * (d.x - cm1 - (yv.x - cmean) * cim2);
                d.y = ca * (d.y - cm1 - (yv.y - cmean) * cim2);
                d.z = ca * (d.z - cm1 - (yv.z - cmean) * cim2);
                d.w = ca * (d.w - cm1 - (yv.w - cmean) * cim2);
                dr[q] = d;
            }
        }
        __syncthreads();
    }

    for (int c = warp; c < C; c += NW) {
        float2 acc[8][7];
#pragma unroll
        for (int o2 = 0; o2 < 8; ++o2)
#pragma unroll
            for (int k = 0; k < 7; ++k) acc[o2][k] = make_float2(0.f, 0.f);
        const float* xr = xs + c * XS;
#pragma unroll 2
        for (int ll = lane; ll < CH; ll += 32) {
            float2 d2[8];
#pragma unroll
            for (int o2 = 0; o2 < 8; ++o2) d2[o2] = make_float2(dys[(2 * o2) * CH + ll], dys[(2 * o2 + 1) * CH + ll]);
            float xw[8];        // x[c][2 l + k - 3] = xs[2 ll + k + 1]
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float2 v = *reinterpret_cast<const float2*>(xr + 2 * ll + 2 * q);
                xw[2 * q] = v.x; xw[2 * q + 1] = v.y;
            }
#pragma unroll
            for (int k = 0; k < 7; ++k) {
                const float2 xv = bc2(xw[k + 1]);
#pragma unroll
                for (int o2 = 0; o2 < 8; ++o2) acc[o2][k] = __ffma2_rn(d2[o2], xv, acc[o2][k]);
            }
        }
        // sum over the 32 lanes: 112 values a[o * 7 + k]; after four halvings (112 -> 7) the lanes 2o, 2o + 1 hold the two halves
        // of output channel o
        float a[112];
#pragma unroll
        for (int o2 = 0; o2 < 8; ++o2)
#pragma unroll
            for (int k = 0; k < 7; ++k) { a[(2 * o2) * 7 + k] = acc[o2][k].x; a[(2 * o2 + 1) * 7 + k] = acc[o2][k].y; }
        int n = 112;
#pragma unroll
        for (int msk = 16; msk >= 2; msk >>= 1) {
            n >>= 1;
            const bool upper = (lane & msk) != 0;
#pragma unroll
            for (int i = 0; i < 56; ++i) {
                if (i < n) {
                    const float keep = upper ? a[i + n] : a[i];
                    const float send = upper ? a[i] : a[i + n];
                    a[i] = keep + __shfl_xor_sync(0xffffffffu, send, msk);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 7; ++k) a[k] += __shfl_xor_sync(0xffffffffu, a[k], 1);
        if ((lane & 1) == 0) {
            const int o = lane >> 1;
#pragma unroll
            for (int k = 0; k < 7; ++k) s_G[(c * 16 + o) * 7 + k] = a[k];
        }
    }
    __syncthreads();
    const int NG = C * 112;
    if (NCH > 1) {
        float* mine = gp + ((size_t)b * NCH + chunk) * NG;
        for (int e = tid; e < NG; e += NT) mine[e] = s_G[e];
        __threadfence();
        __syncthreads();
        if (tid == 0) s_last = atomicAdd(counter + b, 1) == NCH - 1;
        __syncthreads();
        if (!s_last) return;
        __threadfence();
        for (int e = tid; e < NG; e += NT) {         // fixed order of the chunks: the row's G does not depend on which CTA came last
            float G = 0.f;
            for (int r = 0; r < NCH; ++r) G += r == chunk ? s_G[e] : __ldcg(gp + ((size_t)b * NCH + r) * NG + e);
            s_G[e] = G;
        }
        __syncthreads();
    }
    // the row is complete: weight gradient, gate gradient, ChannelAttention parameter gradients (reverse of models.py:28-31)
    for (int e = tid; e < NG; e += NT) {
        const int c = e / 112, rem = e - c * 112, o = rem / 7, k = rem - o * 7;
        const float g = gate ? __ldg(gate + b * C + c) : 1.f;
        atomicAdd(dw + (o * C + c) * 7 + k, g * s_G[e]);
    }
    if (!gate || A <= 0) return;
    for (int c = warp; c < C; c += NW) {
        float s = 0.f;
        for (int r = lane; r < 112; r += 32) {
            const int o = r / 7, k = r - o * 7;
            s = fmaf(__ldg(w + (o * C + c) * 7 + k), s_G[c * 112 + r], s);
        }
        s = warp_sum(s);
        if (lane == 0) s_dgr[c] = s;
    }
    __syncthreads();
    if (tid < C) {
        const float g = __ldg(gate + b * C + tid);
        s_dg[tid] = s_dgr[tid] * g * (1.f - g);               // d(pre-sigmoid)
    }
    __syncthreads();
    if (tid < A) {
        float hsum = 0.f, dh = 0.f;
        for (int c = 0; c < C; ++c) {
            hsum += __ldg(ca_w1 + tid * C + c) * __ldg(mean + b * C + c);
            dh += s_dg[c] * __ldg(ca_w2 + c * A + tid);
        }
        const float hr = fmaxf(hsum, 0.f);
        s_hid[tid] = hr;
        s_dh[tid] = hr > 0.f ? dh : 0.f;
    }
    __syncthreads();
    for (int e = tid; e < C * A; e += NT) {
        const int c2 = e / A, a2 = e - c2 * A;        // dw2[c2, a2]
        const int a1 = e / C, c1 = e - a1 * C;        // dw1[a1, c1]
        atomicAdd(dca_w2 + e, s_dg[c2] * s_hid[a2]);
        atomicAdd(dca_w1 + e, s_dh[a1] * __ldg(mean + b * C + c1));
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------
constexpr int C1B_MAX_CHUNKS = 16;
constexpr size_t C1B_MAX_SMEM = 200 * 1024;

// chunk length of conv1_bwd for rows of L1 = T / 2 positions: a multiple of 32 near `want`, at most C1B_MAX_CHUNKS chunks per row,
// tiles within C1B_MAX_SMEM.  Returns false when no such chunk exists (very long sequences: the separate kernels take over).
static bool conv1_bwd_plan(int C, int L1, int* CH, int* NCH) {
    const int want = option_get("CONV1_BWD_CH", 480);
    int ch = want < 32 ? 32 : (want / 32) * 32;
    const int whole = ((L1 + 31) / 32) * 32;
    if (ch > whole) ch = whole;
    while (cdiv(L1, ch) > C1B_MAX_CHUNKS) ch += 32;
    if ((size_t)(C * (2 * ch + 8) + 32 * ch + C * 112) * sizeof(float) > C1B_MAX_SMEM) return false;
    *CH = ch;
    *NCH = cdiv(L1, ch);
    return true;
}

bool conv_bwd_supported(const float* x, int C, int T, int O) {
    // T % 64 == 0: the conv2 output rows (T / 8 floats) are handled in groups of 8 elements / 16-byte pieces everywhere
    if ((reinterpret_cast<uintptr_t>(x) & 15) || T % 64 != 0 || T < 64 || C < 1 || C > 16 || O != C2B_CO) return false;
    int ch, nch;
    return conv1_bwd_plan(C, T / 2, &ch, &nch);
}

// scratch floats of launch_conv2_bwd / launch_conv1_bwd for a batch of B rows (independent of run-time options)
int64_t conv2_bwd_scratch_floats(int B, int P1) { return (int64_t)B * cdiv(conv_out_len(P1, CONV2_K, CONV2_S, CONV2_P), C2B_TM) * C2B_NW; }
int64_t conv1_bwd_scratch_floats(int B, int C) { return (int64_t)B * C1B_MAX_CHUNKS * C * 112; }

int launch_pool_bwd_tm(const float* y, const double* stats, const float* gamma, const float* beta, const float* rm, const float* rv,
                       const float* dout, int B, int C, int Lin, int training, float* dy, double* red, cudaStream_t st, int Bstat) {
    MMS_REQUIRE((C == 16 || C == 32 || C == 64) && Lin % 8 == 0, "pool_bwd_tm: unsupported shape (C %d, L %d)", C, Lin);
    const int Lout = pool_out_len(Lin);
    if (Bstat <= 0) Bstat = B;
    const int NS = 256 / C;
    const int iters = option_get("POOL_TM_ITERS", 2) >= 4 ? 4 : 2;
    dim3 grid(cdiv(Lin, 8 * NS * iters), B);
    MMS_PROF_BEGIN(st);
#define MMS_POOL_TM(CC, IT) MMS_LAUNCH((pool_bwd_tm_kernel<CC, IT>), grid, dim3(256), 0, st, y, stats, gamma, beta, rm, rv, dout, Bstat, Lin, Lout, training, dy, red)
    if (C == 16) { if (iters == 4) MMS_POOL_TM(16, 4); else MMS_POOL_TM(16, 2); }
    else if (C == 32) { if (iters == 4) MMS_POOL_TM(32, 4); else MMS_POOL_TM(32, 2); }
    else { if (iters == 4) MMS_POOL_TM(64, 4); else MMS_POOL_TM(64, 2); }
#undef MMS_POOL_TM
    MMS_LAUNCH_CHECK("pool_bwd_tm_kernel");
    return MMS_OK;
}

int launch_pool_bwd_ncl(const float* y, const double* stats, const float* gamma, const float* beta, const float* rm, const float* rv,
                        const float* dout, int B, int C, int Lin, int training, float* dy, double* red, cudaStream_t st, int Bstat) {
    const int Lout = pool_out_len(Lin);
    MMS_REQUIRE(Lin % 8 == 0 && Lout % 4 == 0 && ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(dout) | reinterpret_cast<uintptr_t>(dy)) & 15) == 0,
                "pool_bwd_ncl: unsupported shape / alignment (L %d)", Lin);
    if (Bstat <= 0) Bstat = B;
    dim3 grid(cdiv(Lin, 2048), C, B);
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(pool_bwd_ncl_kernel, grid, dim3(256), 0, st, y, stats, gamma, beta, rm, rv, dout, Bstat, C, Lin, Lout, training, dy, red);
    MMS_LAUNCH_CHECK("pool_bwd_ncl_kernel");
    return MMS_OK;
}

static const BnBwd kNoBn = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, 1.f};

// Both gradients of conv2 (C_out = 32).  dp1 [B,16,P1] is written (dp1 == nullptr: the weight gradient alone); dw (+=) receives the weight gradient through `scratch`
// (conv2_bwd_scratch_floats) and launch_wgrad_reduce.  w: the weights in conv2_w_relayout_kernel's order.
int launch_conv2_w_relayout(const float* w, float* wd, cudaStream_t st) {
    MMS_PROF_BEGIN(st);
    conv2_w_relayout_kernel<<<cdiv(C2B_NW, 256), 256, 0, st>>>(w, C2B_NW, wd);
    MMS_LAUNCH_CHECK("conv2_w_relayout_kernel");
    return MMS_OK;
}
int64_t conv2_w_relayout_floats() { return C2B_NW; }

int launch_conv2_bwd(const float* dyn, const float* w, const float* p1, int B, int P1, float* dp1, float* scratch, cudaStream_t st,
                     const BnBwd* bnp) {
    const BnBwd& bn = bnp ? *bnp : kNoBn;
    const int Lout = conv_out_len(P1, CONV2_K, CONV2_S, CONV2_P);
    MMS_REQUIRE(P1 % 4 == 0 && Lout % 4 == 0, "conv2_bwd: lengths %d / %d must be multiples of 4", P1, Lout);
    MMS_REQUIRE(((reinterpret_cast<uintptr_t>(dyn) | reinterpret_cast<uintptr_t>(p1) | reinterpret_cast<uintptr_t>(dp1) |
                  reinterpret_cast<uintptr_t>(scratch) | reinterpret_cast<uintptr_t>(bn.y) | reinterpret_cast<uintptr_t>(w)) & 15) == 0, "conv2_bwd: operands must be 16-byte aligned");
    const size_t smem = (size_t)C2B_SMEM_FLOATS * sizeof(float);
    static PerDeviceOnce attr_once;
    if (attr_once.need()) {
        MMS_CUDA(cudaFuncSetAttribute(conv2_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        MMS_CUDA(cudaFuncSetAttribute(conv2_wgrad_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    dim3 grid(cdiv(Lout, C2B_TM), B);
    MMS_PROF_BEGIN(st);
    if (dp1) {
        MMS_LAUNCH(conv2_bwd_kernel, grid, dim3(128), smem, st, dyn, w, p1, dp1, scratch, P1, Lout, bn);
        MMS_LAUNCH_CHECK("conv2_bwd_kernel");
    } else {        // stage 1 frozen: the weight gradient alone
        MMS_LAUNCH(conv2_wgrad_bwd_kernel, grid, dim3(128), smem, st, dyn, w, p1, scratch, P1, Lout, bn);
        MMS_LAUNCH_CHECK("conv2_wgrad_bwd_kernel");
    }
    return MMS_OK;
}

// dw[0, n) += sum over the `parts` partial gradients in scratch
int launch_wgrad_reduce(const float* scratch, int parts, int n, float* dw, cudaStream_t st) {
    int S = parts < 16 ? parts : 16;
    if (S < 1) S = 1;
    MMS_PROF_BEGIN(st);
    wgrad_reduce_kernel<<<dim3(cdiv(n, 256), S), 256, 0, st>>>(scratch, parts, n, dw);
    MMS_LAUNCH_CHECK("wgrad_reduce_kernel");
    return MMS_OK;
}
int conv2_bwd_parts(int B, int P1) { return B * cdiv(conv_out_len(P1, CONV2_K, CONV2_S, CONV2_P), C2B_TM); }

// Weight gradient of conv1 (dw +=) and -- with gate != nullptr -- the ChannelAttention parameter gradients (dca_w1, dca_w2 +=).
// counter: B ints, zero on entry.
int launch_conv1_bwd(const float* x, const float* dyn, const float* w, const float* gate, const float* mean, const float* ca_w1,
                     const float* ca_w2, int B, int C, int T, float* scratch, int* counter, float* dw, float* dca_w1, float* dca_w2,
                     cudaStream_t st, const BnBwd* bnp) {
    const BnBwd& bn = bnp ? *bnp : kNoBn;
    MMS_REQUIRE(T % 8 == 0 && C >= 1 && C <= 16, "conv1_bwd: unsupported shape (C %d, T %d)", C, T);
    MMS_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dyn) | reinterpret_cast<uintptr_t>(bn.y)) & 15) == 0,
                "conv1_bwd: operands must be 16-byte aligned");
    const int L1 = T / 2;
    int CH = 0, NCH = 0;
    MMS_REQUIRE(conv1_bwd_plan(C, L1, &CH, &NCH), "conv1_bwd: sequence length %d too long for the chunked kernel", T);
    const int NW = C <= 8 ? C : (C + 1) / 2;
    const size_t smem = (size_t)(C * (2 * CH + 8) + 32 * CH + C * 112) * sizeof(float);
    static PerDeviceOnce attr_once;
    if (attr_once.need()) MMS_CUDA(cudaFuncSetAttribute(conv1_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C1B_MAX_SMEM));
    MMS_PROF_BEGIN(st);
    MMS_LAUNCH(conv1_bwd_kernel, dim3(NCH, B), dim3(32 * NW), smem, st, x, dyn, w, gate, mean, ca_w1, ca_w2, C, C / 4, T, L1, CH, scratch,
               counter, dw, dca_w1, dca_w2, bn);
    MMS_LAUNCH_CHECK("conv1_bwd_kernel");
    return MMS_OK;
}

}  // namespace mms
