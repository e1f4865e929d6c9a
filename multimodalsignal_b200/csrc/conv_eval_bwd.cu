// Input gradient of an eval-mode forward (mms_cnngru_input_gradient): the kernels that only this path runs.
// In eval mode BatchNorm is the per-channel affine map a*y + b of the running statistics, so the backward of
// MaxPool(ReLU(BN(y))) needs no batch reduction: every element's gradient is a * (its pool-window share of the upstream
// gradient, if it won its window and is positive).  That lets one launch go from the GRU's input gradient d(seq) to
// conv1's output gradient dy1:
//   encoder_eval_bwd_kernel : stage-2 pool/ReLU/BN backward -> conv2 input gradient -> stage-1 pool/ReLU/BN backward,
//                             one CTA per (window, TJ pool-1 positions), every intermediate in shared memory;
//   attn_input_grad_kernel  : ChannelAttention's share of dx -- gate gradient -> mean gradient, broadcast as 1/T --
//                             applied to conv1's input gradient in place (no parameter gradient);
//   head_input_grad_kernel  : d(classifier hidden layer) from dlogits (no weight gradient).
#include "conv_common.cuh"

namespace mms {

constexpr int ATTN_MAX_A = 4;     // in_channels <= 16: at most 4 hidden units in the gate MLP

__device__ __forceinline__ int floor_half(int a) { return a >= 0 ? a / 2 : -((-a + 1) / 2); }

// d(maxpool(3,2,1) of relu(z)) at element i of a row of Lin elements, from the upstream gradient d(j) of the Lout windows.
// Same winner rule and summation order as pool_relu_bwd_kernel: the first maximal element of a window wins (ATen).
template <typename ZF, typename DF>
__device__ __forceinline__ float pool_relu_grad(const ZF& z, const DF& d, int i, int Lin, int Lout) {
    const float zi = z(i);
    float dsum = 0.f;
    if ((i & 1) == 0) {
        const int j = i >> 1;
        const bool left_wins = i - 1 >= 0 && z(i - 1) >= zi;
        const bool right_wins = i + 1 < Lin && z(i + 1) > zi;
        if (j < Lout && !left_wins && !right_wins) dsum += d(j);
    } else {
        const int ja = (i + 1) >> 1;
        if (ja < Lout) {
            const bool lose = (i + 1 < Lin && z(i + 1) > zi) || (i + 2 < Lin && z(i + 2) > zi);
            if (!lose) dsum += d(ja);
        }
        const int jb = (i - 1) >> 1;
        if (jb < Lout) {
            const bool lose = (i - 2 >= 0 && z(i - 2) >= zi) || z(i - 1) >= zi;
            if (!lose) dsum += d(jb);
        }
    }
    return zi > 0.f ? dsum : 0.f;
}

// One CTA = window b x pool-1 positions [J0, J0 + TJ).  It writes dy1 at conv1 positions [2 J0, 2 J0 + 2 TJ), which need
// d(p1) at the TJ + 1 positions [J0, J0 + TJ]; those need dy2 at NL2 conv2 positions from L0 = J0/2 - 1, and those the
// stage-2 pool gradient d(seq) of NQ windows from Q0.  Every tensor is read from global memory once per CTA (y1 / y2
// neighbours come through L1), nothing but dy1 is written.  grid = (cdiv(P1, TJ), B), block = NT.
template <int CO, int TJ, int NT>
__global__ void __launch_bounds__(NT) encoder_eval_bwd_kernel(const float* __restrict__ dseq, const float* __restrict__ y2,
                                                              const float* __restrict__ y1, const float* __restrict__ w2,
                                                              const float* __restrict__ g1, const float* __restrict__ b1,
                                                              const float* __restrict__ rm1, const float* __restrict__ rv1,
                                                              const float* __restrict__ g2, const float* __restrict__ b2,
                                                              const float* __restrict__ rm2, const float* __restrict__ rv2,
                                                              int L1c, int P1, int L2c, int L, float* __restrict__ dy1) {
    constexpr int CI = CONV2_CI, KW = CONV2_K;
    constexpr int NJ = TJ + 1;
    constexpr int NL2 = TJ / 2 + 3;
    constexpr int NQ = NL2 / 2 + 3;
    static_assert(TJ % 2 == 0 && TJ <= NT && 2 * NT >= TJ && CO + CI <= NT, "encoder_eval_bwd: bad tiling");
    extern __shared__ __align__(16) float smem[];
    float* ws = smem;                       // [KW][CO][CI]  conv2 weights
    float* dys = ws + KW * CO * CI;         // [CO][NL2]     dy2
    float* dq = dys + CO * NL2;             // [NQ][CO]      d(seq), time-major like its source
    float* dps = dq + NQ * CO;              // [CI][NJ]      d(p1)
    __shared__ float s_a2[CO], s_b2[CO], s_a1[CI], s_b1[CI];

    const int b = blockIdx.y, J0 = blockIdx.x * TJ, tid = threadIdx.x;
    const int L0 = J0 / 2 - 1;
    const int Q0 = floor_half(L0 - 1);
    if (tid < CO) {
        const BnAffine af = bn_affine(0, nullptr, g2, b2, rm2, rv2, tid, CO, 1.0);
        s_a2[tid] = af.a; s_b2[tid] = af.b;
    } else if (tid < CO + CI) {
        const BnAffine af = bn_affine(0, nullptr, g1, b1, rm1, rv1, tid - CO, CI, 1.0);
        s_a1[tid - CO] = af.a; s_b1[tid - CO] = af.b;
    }
    // the NQ rows of d(seq) are one contiguous run of the time-major tensor
    const float* dsb = dseq + (size_t)b * L * CO + (int64_t)Q0 * CO;
    for (int idx = tid; idx < NQ * CO; idx += NT) {
        const int q = Q0 + idx / CO;
        dq[idx] = q >= 0 && q < L ? __ldg(dsb + idx) : 0.f;
    }
    for (int idx = tid; idx < KW * CO * CI; idx += NT) {
        const int c = idx % CI, ko = idx / CI, o = ko % CO, k = ko / CO;
        ws[idx] = __ldg(w2 + ((size_t)o * CI + c) * KW + k);
    }
    __syncthreads();

    // dy2 = a2 * d(pool2(relu(bn2(y2)))) at positions L0 + [0, NL2)
    const float* y2b = y2 + (size_t)b * CO * L2c;
    for (int idx = tid; idx < CO * NL2; idx += NT) {
        const int o = idx / NL2, l = L0 + (idx - o * NL2);
        float v = 0.f;
        if (l >= 0 && l < L2c) {
            const float* row = y2b + (size_t)o * L2c;
            const float a = s_a2[o], sh = s_b2[o];
            const auto z = [&](int i) { return fmaxf(fmaf(a, __ldg(row + i), sh), 0.f); };
            const auto d = [&](int j) { return dq[(j - Q0) * CO + o]; };
            v = a * pool_relu_grad(z, d, l, L2c, L);
        }
        dys[idx] = v;
    }
    __syncthreads();

    // d(p1)[c, j] = sum_{o, k : 2 l + k - 2 = j} w2[o, c, k] dy2[o, l].  Only the taps k = j (mod 2) contribute: the first
    // half of the threads takes the even positions, the second half the odd ones, so that no warp diverges on the tap count.
    for (int r = tid; r < NJ; r += NT) {
        const int jj = r < TJ ? (r < TJ / 2 ? 2 * r : 2 * (r - TJ / 2) + 1) : r;
        const int j = J0 + jj;
        float acc[CI];
#pragma unroll
        for (int c = 0; c < CI; ++c) acc[c] = 0.f;
        for (int k = jj & 1; k < KW; k += 2) {
            const int ll = (jj + 2 - k) / 2 + 1;          // jj + 2 - k is even and >= -2
            for (int o = 0; o < CO; ++o) {
                const float dv = dys[o * NL2 + ll];
                const float4* wv = reinterpret_cast<const float4*>(ws + (k * CO + o) * CI);
#pragma unroll
                for (int c4 = 0; c4 < CI / 4; ++c4) {
                    const float4 wq = wv[c4];
                    acc[4 * c4 + 0] = fmaf(wq.x, dv, acc[4 * c4 + 0]);
                    acc[4 * c4 + 1] = fmaf(wq.y, dv, acc[4 * c4 + 1]);
                    acc[4 * c4 + 2] = fmaf(wq.z, dv, acc[4 * c4 + 2]);
                    acc[4 * c4 + 3] = fmaf(wq.w, dv, acc[4 * c4 + 3]);
                }
            }
        }
        const bool valid = j < P1;
#pragma unroll
        for (int c = 0; c < CI; ++c) dps[c * NJ + jj] = valid ? acc[c] : 0.f;
    }
    __syncthreads();

    // dy1 = a1 * d(pool1(relu(bn1(y1)))) at conv1 positions [2 J0, 2 J0 + 2 TJ)
    const float* y1b = y1 + (size_t)b * CI * L1c;
    float* dy1b = dy1 + (size_t)b * CI * L1c;
    const int i0 = 2 * J0;
    for (int idx = tid; idx < CI * 2 * TJ; idx += NT) {
        const int c = idx / (2 * TJ), i = i0 + (idx - c * 2 * TJ);
        if (i >= L1c) continue;
        const float* row = y1b + (size_t)c * L1c;
        const float a = s_a1[c], sh = s_b1[c];
        const auto z = [&](int t) { return fmaxf(fmaf(a, __ldg(row + t), sh), 0.f); };
        const auto d = [&](int jw) { return dps[c * NJ + (jw - J0)]; };
        dy1b[(size_t)c * L1c + i] = a * pool_relu_grad(z, d, i, L1c, P1);
    }
}

// dx[b,c,t] = dxg[b,c,t] * gate[b,c] + ds[b,c] / T in place, where dxg is conv1's input gradient (the gradient of x * gate)
// and ds the gradient that reaches mean[b,c] through the gate MLP from dgate[b,c] = sum_t dxg * x.  Each CTA forms ds for its
// own row (A = C/4 <= 4 hidden units: a few dozen FMAs) with the arithmetic of chan_param_bwd_kernel.  A = 0 (C < 4): the gate
// is the constant sigmoid(0) and ds = 0.  grid = (cdiv(T, 1024), B * C), block = 256.
__global__ void __launch_bounds__(256) attn_input_grad_kernel(const float* __restrict__ dgate, const float* __restrict__ mean,
                                                              const float* __restrict__ gate, const float* __restrict__ w1,
                                                              const float* __restrict__ w2, int C, int A, int T,
                                                              float* __restrict__ dx) {
    __shared__ float s_add;
    const int row = blockIdx.y, b = row / C, c = row - b * C;
    if (threadIdx.x == 0) {
        float dh[ATTN_MAX_A], h[ATTN_MAX_A];
#pragma unroll
        for (int a = 0; a < ATTN_MAX_A; ++a) {
            float s = 0.f;
            if (a < A)
                for (int cc = 0; cc < C; ++cc) s += w1[a * C + cc] * mean[b * C + cc];
            h[a] = fmaxf(s, 0.f);
            dh[a] = 0.f;
        }
        for (int cc = 0; cc < C; ++cc) {
            const float g = gate[b * C + cc];
            const float dp = dgate[b * C + cc] * g * (1.f - g);
#pragma unroll
            for (int a = 0; a < ATTN_MAX_A; ++a)
                if (a < A) dh[a] += dp * w2[cc * A + a];
        }
        float s = 0.f;
#pragma unroll
        for (int a = 0; a < ATTN_MAX_A; ++a)
            if (a < A) s += (h[a] > 0.f ? dh[a] : 0.f) * w1[a * C + c];
        s_add = A > 0 ? s / (float)T : 0.f;
    }
    __syncthreads();
    const float g = gate[row], add = s_add;
    const size_t base = (size_t)row * T;
    for (int t = blockIdx.x * 1024 + threadIdx.x; t < min(T, (blockIdx.x + 1) * 1024); t += blockDim.x)
        dx[base + t] = dx[base + t] * g + add;
}

// dhid[b,i] = relu'(hid[b,i]) * sum_c dlogits[b,c] w3[c,i] (eval mode: no dropout).  grid = cdiv(B * 64, 256), block = 256.
__global__ void __launch_bounds__(256) head_input_grad_kernel(const float* __restrict__ hid, const float* __restrict__ dlogits,
                                                              const float* __restrict__ w3, int B, int nc,
                                                              float* __restrict__ dhid) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * HEAD_HID) return;
    const int b = e / HEAD_HID, i = e - b * HEAD_HID;
    float dhd = 0.f;
    for (int c = 0; c < nc; ++c) dhd = fmaf(dlogits[(size_t)b * nc + c], __ldg(w3 + c * HEAD_HID + i), dhd);
    dhid[e] = hid[e] > 0.f ? dhd : 0.f;
}

// ---- launchers -------------------------------------------------------------------------------
constexpr int ENC_EVAL_TJ = 256, ENC_EVAL_NT = 256;

template <int CO>
static int encoder_eval_bwd_launch(const float* dseq, const float* y2, const float* y1, const float* w2, const float* g1,
                                   const float* b1, const float* rm1, const float* rv1, const float* g2, const float* b2,
                                   const float* rm2, const float* rv2, int B, int L1c, float* dy1, cudaStream_t st) {
    constexpr int TJ = ENC_EVAL_TJ, NT = ENC_EVAL_NT;
    constexpr int NL2 = TJ / 2 + 3, NQ = NL2 / 2 + 3;
    const int P1 = pool_out_len(L1c);
    const int L2c = conv_out_len(P1, CONV2_K, CONV2_S, CONV2_P);
    const int L = pool_out_len(L2c);
    const size_t smem = (size_t)(CONV2_K * CO * CONV2_CI + CO * NL2 + NQ * CO + CONV2_CI * (TJ + 1)) * sizeof(float);
    auto kern = encoder_eval_bwd_kernel<CO, TJ, NT>;
    static PerDeviceOnce attr_once;
    if (attr_once.need()) { MMS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); }
    dim3 grid(cdiv(P1, TJ), B);
    MMS_PROF_BEGIN(st);
    kern<<<grid, NT, smem, st>>>(dseq, y2, y1, w2, g1, b1, rm1, rv1, g2, b2, rm2, rv2, L1c, P1, L2c, L, dy1);
    MMS_LAUNCH_CHECK("encoder_eval_bwd_kernel");
    return MMS_OK;
}

// dy1 [B, 16, L1c] from d(seq) [B, L, O] (time-major) after an eval-mode forward; bn = [rm1 | rv1 | rm2 | rv2].
int launch_encoder_eval_bwd(const float* dseq, const float* y2, const float* y1, const float* w2, const float* g1,
                            const float* b1, const float* g2, const float* b2, const float* bn, int B, int O, int L1c,
                            float* dy1, cudaStream_t st) {
    const float *rm1 = bn, *rv1 = bn + CONV1_CO, *rm2 = bn + 2 * CONV1_CO, *rv2 = bn + 2 * CONV1_CO + O;
    if (O == 16) return encoder_eval_bwd_launch<16>(dseq, y2, y1, w2, g1, b1, rm1, rv1, g2, b2, rm2, rv2, B, L1c, dy1, st);
    if (O == 32) return encoder_eval_bwd_launch<32>(dseq, y2, y1, w2, g1, b1, rm1, rv1, g2, b2, rm2, rv2, B, L1c, dy1, st);
    MMS_REQUIRE(O == 64, "encoder_eval_bwd: cnn_out %d not in {16,32,64}", O);
    return encoder_eval_bwd_launch<64>(dseq, y2, y1, w2, g1, b1, rm1, rv1, g2, b2, rm2, rv2, B, L1c, dy1, st);
}

int launch_attn_input_grad(const float* dgate, const float* mean, const float* gate, const float* w1, const float* w2, int B,
                           int C, int T, float* dx, cudaStream_t st) {
    const int A = C / 4;
    MMS_REQUIRE(A <= ATTN_MAX_A, "attn_input_grad: %d channels", C);
    dim3 grid(cdiv(T, 1024), B * C);
    MMS_PROF_BEGIN(st);
    attn_input_grad_kernel<<<grid, 256, 0, st>>>(dgate, mean, gate, w1, w2, C, A, T, dx);
    MMS_LAUNCH_CHECK("attn_input_grad_kernel");
    return MMS_OK;
}

int launch_head_input_grad(const float* hid, const float* dlogits, const float* w3, int B, int nc, float* dhid, cudaStream_t st) {
    MMS_PROF_BEGIN(st);
    head_input_grad_kernel<<<cdiv((int64_t)B * HEAD_HID, 256), 256, 0, st>>>(hid, dlogits, w3, B, nc, dhid);
    MMS_LAUNCH_CHECK("head_input_grad_kernel");
    return MMS_OK;
}

}  // namespace mms
