// Epoch plumbing that the reference does on the host, moved onto the device so that a training
// step needs no host work besides one CUDA-graph replay and an evaluation pass one read-back:
//   * batch assembly of a shuffling DataLoader (reference trainer.py:130,140-142 iterating
//     DataLoader(train_dataset, batch_size, shuffle=True), main.py:111) as an index gather driven by a
//     device-resident permutation and a device-resident cursor;
//   * the evaluation bookkeeping of trainer.py:217-228 (loss.item() * batch accumulation,
//     softmax -> argmax, the prediction / label lists that feed sklearn's accuracy_score and
//     f1_score) as one kernel: summed loss in float64, predictions, and the confusion matrix the two
//     metrics are functions of.
// Both are HBM-streaming / latency-trivial kernels; integer results are exact.
#include "mms_common.cuh"

namespace mms {

constexpr int MAX_NC = 8;      // as in head_opt.cu (mms_cnngru_desc.num_classes <= 8)

// out_x[b, :] = data[perm[cursor + b], :] (rows of row_f4 float4), out_y[b] = labels[perm[cursor + b]].
// grid = (chunks, B).  With `advance` the last CTA to finish moves the cursor by B (every CTA has read
// it by then), so consecutive graph replays walk through the permutation without host involvement.
__global__ void __launch_bounds__(256) batch_gather_kernel(const float4* __restrict__ data, const int64_t* __restrict__ labels,
                                                           const int64_t* __restrict__ perm, int64_t* cursor, int64_t n_rows,
                                                           int64_t row_f4, float4* __restrict__ out_x, int64_t* __restrict__ out_y,
                                                           int advance, int32_t* scratch) {
    MMS_PDL_PROLOGUE();
    const int b = blockIdx.y;
    const int64_t base = cursor ? *cursor : 0;
    int64_t src = perm ? perm[base + b] : base + b;
    src = src < 0 ? 0 : (src >= n_rows ? n_rows - 1 : src);        // never read outside the dataset
    const float4* s = data + src * row_f4;
    float4* o = out_x + (int64_t)b * row_f4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < row_f4; i += (int64_t)gridDim.x * blockDim.x) o[i] = __ldg(s + i);
    if (blockIdx.x == 0 && threadIdx.x == 0 && out_y) out_y[b] = labels[src];
    if (advance) {
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            const int total = (int)(gridDim.x * gridDim.y);
            if (atomicAdd(scratch, 1) == total - 1) {
                *cursor = base + gridDim.y;
                *scratch = 0;
            }
        }
    }
}

// Row b's loss term lse - logit[y] (y clamped into [0, nc)), its first arg-max and its clamped label.
__device__ __forceinline__ float eval_row(const float* __restrict__ logits, const int64_t* __restrict__ labels, int b, int nc,
                                          int* am_out, int* y_out) {
    float v[MAX_NC];
    for (int c = 0; c < nc; ++c) v[c] = logits[(size_t)b * nc + c];
    float mx = v[0];
    int am = 0;
    for (int c = 1; c < nc; ++c)              // first maximum; a NaN counts as the maximum, like torch.argmax
        if (!(mx != mx) && (v[c] > mx || v[c] != v[c])) { mx = v[c]; am = c; }
    float m2 = -INFINITY;
    for (int c = 0; c < nc; ++c) m2 = fmaxf(m2, v[c]);
    float se = 0.f;
    for (int c = 0; c < nc; ++c) se += expf(v[c] - m2);
    const float lse = m2 + logf(se);
    int y = (int)labels[b];
    y = y < 0 ? 0 : (y >= nc ? nc - 1 : y);
    *am_out = am;
    *y_out = y;
    return lse - v[y];
}

// Single CTA.  For every row: loss_sum += lse - logit[y] (float64), pred = first arg-max of the logits
// (== torch.argmax(softmax(logits)), ties to the lowest index), conf[y * nc + pred] += 1.
// With class_weight (CrossEntropyLoss(weight=w)) the loss is the reference's per-loader-batch accumulation instead: the rows
// are taken in groups of `group` consecutive rows, each reduced over the block in a fixed order, and group g adds
// n_g * sum w[y] l / sum w[y] (the groups in order).  A null class_weight runs exactly the unweighted code.
__global__ void __launch_bounds__(256) eval_accumulate_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                                                              int B, int nc, int64_t* __restrict__ preds, int64_t* conf,
                                                              double* loss_sum, const float* __restrict__ class_weight, int group) {
    __shared__ double s_part[8];
    __shared__ double s_wpart[8];
    __shared__ unsigned int s_conf[MAX_NC * MAX_NC];
    for (int i = threadIdx.x; i < nc * nc; i += blockDim.x) s_conf[i] = 0u;
    __syncthreads();
    double local = 0.0;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        int am, y;
        const float l = eval_row(logits, labels, b, nc, &am, &y);
        local += (double)l;
        if (preds) preds[b] = am;
        atomicAdd(&s_conf[y * nc + am], 1u);
    }
    if (class_weight) {
        double total = 0.0;                                  // meaningful in thread 0 only
        for (int g0 = 0; g0 < B; g0 += group) {
            const int n = B - g0 < group ? B - g0 : group;
            double num = 0.0, den = 0.0;
            for (int b = g0 + threadIdx.x; b < g0 + n; b += blockDim.x) {
                int am, y;
                const float l = eval_row(logits, labels, b, nc, &am, &y);
                const double wy = (double)class_weight[y];
                num += wy * (double)l;
                den += wy;
            }
            num = warp_sum(num);
            den = warp_sum(den);
            if ((threadIdx.x & 31) == 0) { s_part[threadIdx.x >> 5] = num; s_wpart[threadIdx.x >> 5] = den; }
            __syncthreads();
            if (threadIdx.x == 0) {
                double sn = 0.0, sd = 0.0;
                for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { sn += s_part[w]; sd += s_wpart[w]; }
                total += (double)n * (sn / sd);
            }
            __syncthreads();
        }
        if (threadIdx.x == 0 && loss_sum) *loss_sum += total;
    } else {
        local = warp_sum(local);
        if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = local;
        __syncthreads();
        if (threadIdx.x == 0 && loss_sum) {
            double s = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += s_part[w];
            *loss_sum += s;
        }
    }
    if (conf)
        for (int i = threadIdx.x; i < nc * nc; i += blockDim.x) conf[i] += (int64_t)s_conf[i];
}

}  // namespace mms

using namespace mms;

extern "C" int mms_batch_gather(const float* data, const int64_t* labels, const int64_t* perm, int64_t* cursor_dev, int64_t n_rows,
                                int64_t row_floats, int32_t batch, float* out_x, int64_t* out_y, int32_t advance,
                                int32_t* scratch_dev, mms_stream_t stream) {
    MMS_REQUIRE(data && out_x && batch > 0 && n_rows > 0 && row_floats > 0, "batch_gather: bad arguments");
    MMS_REQUIRE(row_floats % 4 == 0 && (reinterpret_cast<uintptr_t>(data) & 15) == 0 && (reinterpret_cast<uintptr_t>(out_x) & 15) == 0,
                "batch_gather: rows must be 16-byte aligned multiples of 4 floats");
    MMS_REQUIRE(!out_y || labels, "batch_gather: out_y needs labels");
    MMS_REQUIRE(!advance || (cursor_dev && scratch_dev), "batch_gather: advance needs cursor_dev and scratch_dev");
    const int64_t row_f4 = row_floats / 4;
    int chunks = cdiv(row_f4, 256 * 4);
    if (chunks < 1) chunks = 1;
    if (chunks > 64) chunks = 64;
    dim3 grid(chunks, batch);
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    batch_gather_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const float4*>(data), labels, perm, cursor_dev, n_rows, row_f4,
                                              reinterpret_cast<float4*>(out_x), out_y, advance, scratch_dev);
    MMS_LAUNCH_CHECK("batch_gather_kernel");
    return MMS_OK;
}

extern "C" int mms_eval_accumulate(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes, int64_t* preds_out,
                                   int64_t* confusion, double* loss_sum, mms_stream_t stream) {
    MMS_REQUIRE(logits && labels && batch > 0, "eval_accumulate: bad arguments");
    MMS_REQUIRE(num_classes >= 1 && num_classes <= MAX_NC, "eval_accumulate: num_classes %d outside [1,%d]", num_classes, MAX_NC);
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    eval_accumulate_kernel<<<1, 256, 0, st>>>(logits, labels, batch, num_classes, preds_out, confusion, loss_sum, nullptr, batch);
    MMS_LAUNCH_CHECK("eval_accumulate_kernel");
    return MMS_OK;
}

extern "C" int mms_eval_accumulate_weighted(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes,
                                            const float* class_weight, int32_t group, int64_t* preds_out, int64_t* confusion,
                                            double* loss_sum, mms_stream_t stream) {
    MMS_REQUIRE(logits && labels && batch > 0, "eval_accumulate_weighted: bad arguments");
    MMS_REQUIRE(num_classes >= 1 && num_classes <= MAX_NC, "eval_accumulate_weighted: num_classes %d outside [1,%d]", num_classes,
                MAX_NC);
    cudaStream_t st = (cudaStream_t)stream;
    MMS_PROF_BEGIN(st);
    eval_accumulate_kernel<<<1, 256, 0, st>>>(logits, labels, batch, num_classes, preds_out, confusion, loss_sum, class_weight,
                                              group > 0 ? group : batch);
    MMS_LAUNCH_CHECK("eval_accumulate_kernel");
    return MMS_OK;
}
