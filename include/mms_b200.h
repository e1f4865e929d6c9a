/*
 * mms_b200.h -- C ABI of libmms_b200.so: hand-written sm_100a kernels for the hot path of
 * 17LiQi/MultimodalSignal (CnnGruAttentionModel training step + resample/windowing).
 *
 * The reference has no FFI of its own (pure Python / torch.nn, SURVEY.md §8b); the boundary
 * it offers is its Python API.  Every entry point below therefore replaces a *library call
 * site* of the reference, cited as file:line into /root/reference.  The Python host side
 * (the multimodalsignal_b200 package) binds these with ctypes and keeps the reference's class and
 * function signatures.
 *
 * Conventions
 *   - every function returns 0 on success or a negative MMS_E_* code; mms_last_error()
 *     returns a thread-local description of the most recent failure;
 *   - all pointers are DEVICE pointers unless the parameter name ends in _host;
 *   - nothing here allocates, frees or synchronises: workspaces are caller-provided (sizes
 *     from the *_workspace_bytes functions) and every launch goes to the cudaStream_t given
 *     (passed as void* so that this header needs no CUDA headers);
 *   - there is no CPU fallback: mms_init() fails unless the device is compute capability 10.x.
 *   - tensors are contiguous float32 unless stated otherwise.
 */
#ifndef MMS_B200_H
#define MMS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMS_OK 0
#define MMS_E_INVALID (-1)      /* bad argument / unsupported shape            */
#define MMS_E_CUDA (-2)         /* a CUDA runtime call or launch failed        */
#define MMS_E_ARCH (-3)         /* device is not sm_100 (no fallback exists)   */
#define MMS_E_WORKSPACE (-4)    /* workspace too small                         */

typedef void* mms_stream_t;     /* cudaStream_t */

int mms_version(void);
const char* mms_last_error(void);
/* Select `device`, verify it is sm_100 (B200) and raise the dynamic shared-memory limits of
 * the kernels that need it.  Must be called once per process before any other function. */
int mms_init(int device);

/* Diagnostics.  mms_launch_count(): kernels launched by this library since it was loaded
 * (launches recorded into a CUDA graph count once, at capture).  mms_profile_enable(1) makes
 * every subsequent eager launch record a CUDA-event pair on its stream (and clears earlier
 * records); mms_profile_report() synchronises the device and writes one line per kernel name,
 * "name launches total_ms", in first-launch order, into a host buffer. */
int64_t mms_launch_count(void);
int mms_profile_enable(int32_t on);
int mms_profile_report(char* buf_host, int64_t buf_bytes);
/* In-graph timeline (diagnostic; the one place the library allocates: a 16 KB device buffer on first enable).  While
 * enabled, every launch is bracketed by one-thread kernels that store %globaltimer, on the launch's own stream -- also
 * under CUDA-graph capture, where the stamps become graph nodes.  mms_timeline_report() synchronises the device and
 * writes one line per launch of the LAST execution, "name stream_index start_ns end_ns" (relative to the earliest
 * start), into a host buffer.  Enable before capturing / launching, report after; enabling clears earlier records. */
int mms_timeline_enable(int32_t on);
int mms_timeline_report(char* buf_host, int64_t buf_bytes);
/* Weight-gradient kernels normally run on two library-owned side streams (forked from and joined
 * back into the caller's stream, also under CUDA-graph capture).  0 serialises everything on the
 * caller's stream (used while per-kernel times are taken); also MMS_DISABLE_STREAMS=1. */
int mms_set_side_streams(int32_t on);
/* Integer run-time switches for A/B measurements and kernel selection.  mms_set_option("GRU_BWD_RING", 0) has the
 * effect of the environment variable MMS_GRU_BWD_RING=0 but can be changed between launches (the environment is read
 * once, at first use); mms_get_option returns the value in effect (`dflt` if neither was given; defaults are per call
 * site and listed in INTEGRATION.md).  Options never change
 * results beyond the documented tolerances; they select between kernels of this library. */
int mms_set_option(const char* name, int32_t value);
int32_t mms_get_option(const char* name, int32_t dflt);
int mms_clear_option(const char* name);     /* back to the built-in default of every call site */

/* ------------------------------------------------------------------------------------------
 * Model description (reference models.py:39-40 constructor arguments + call-time facts).
 * Conv widths 16 / k7 / k5 and the 64-wide classifier hidden layer are hard-coded in the
 * reference (models.py:46,50,67) and therefore here.
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    int32_t batch;          /* B                                                        */
    int32_t in_channels;    /* C  = len(CHANNELS_TO_USE), main.py:47,116                */
    int32_t seq_len;        /* T  = window samples (3840 @64 Hz, 7680 @128 Hz)          */
    int32_t num_classes;    /* 2 (stress_binary) or 3 (ternary), <= 8                   */
    int32_t cnn_out;        /* cnn_out_channels, models.py:39 (32)                      */
    int32_t hidden;         /* gru_hidden_size: 32, 64 or 128; others are MMS_E_INVALID */
    int32_t layers;         /* gru_num_layers (>= 1)                                    */
    int32_t training;       /* 1: batch-stat BN + dropout (model.train()), 0: eval      */
    int32_t attention;      /* 1: ChannelAttention gate, 0: cnn_gru baseline (SURVEY D3)*/
    int32_t need_grad;      /* 1: keep activations for mms_cnngru_backward              */
    float dropout_p;        /* models.py:40; applied between GRU layers and in the head */
    uint64_t rng_seed;      /* dropout stream seed                                      */
    uint64_t rng_offset;    /* dropout stream offset used when rng_offset_dev == NULL   */
    const int64_t* rng_offset_dev; /* optional device counter read by the kernels
                                      (the fused train step passes its Adam step count) */
    int32_t global_batch;   /* 0 or == batch: single GPU.  > batch: intra-fold data parallelism -- BatchNorm
                               statistics are counted over the global batch (SyncBN) and the BN affine
                               gradients are scaled by batch/global_batch so that a sum all-reduce is exact */
    const float* class_weight; /* NULL: CrossEntropyLoss().  Else float32 [num_classes] device array, the
                                  CrossEntropyLoss(weight=w) of mms_cnngru_train_step (fused and unfused head):
                                  loss = sum_b w[y_b] l_b / sum_b w[y_b], dlogits = w[y_b] (softmax - onehot) / sum_b w[y_b].
                                  The train step needs global_batch == batch; under data parallelism the BN2 sum
                                  vector of mms_cnngru_sync_offsets gets one more double for sum_b w[y_b] */
    uint64_t frozen_segments; /* fine-tuning (requires_grad=False): bit s = segment s of mms_cnngru_param_layout needs
                                 no gradient.  0 = every parameter trains.  See "Frozen segments" below.             */
    const int64_t* adam_ranges_host; /* HOST int64 [adam_nranges][3] = (offset, count, step slot): the flat ranges
                                        mms_cnngru_train_step's Adam updates, one per trainable tensor (see
                                        mms_adam_ranges_step)                                                        */
    int64_t* adam_steps;      /* device int64 step counters indexed by the ranges' step slots.  NULL (with no
                                 table): Adam over the whole buffer with step_dev as the count of every element    */
    int32_t adam_nranges;     /* rows of adam_ranges_host, 0..MMS_MAX_ADAM_RANGES (0: no tensor trains)          */
    const float* clip_max_norm; /* device float32 scalar: mms_cnngru_train_step clips the gradient to this total norm
                                   before Adam (torch.nn.utils.clip_grad_norm_, see "Gradient-norm clipping" below).
                                   NULL: no clipping, and the next two fields are ignored                             */
    double* clip_record;      /* device float64 [5] added to by every clipped step (may be NULL), see mms_grad_norm     */
    void* clip_scratch;       /* device, MMS_GRAD_CLIP_SCRATCH_BYTES, zero-initialised: the step's norm and coefficient */
} mms_cnngru_desc;

/* Flat parameter buffer.  The model's parameters live in ONE float32 buffer so that Adam and
 * the gradient all-reduce are single launches.  Segment order (each segment 16-byte aligned):
 *   0 ca_w1   [C/4, C]      channel_attention.fc.0.weight      models.py:18
 *   1 ca_w2   [C, C/4]      channel_attention.fc.2.weight      models.py:20
 *   2 conv1_w [16, C, 7]    cnn_encoder.0.weight               models.py:46
 *   3 bn1_g [16]  4 bn1_b [16]                                  models.py:47
 *   5 conv2_w [O, 16, 5]    cnn_encoder.4.weight               models.py:50
 *   6 bn2_g [O]   7 bn2_b [O]                                   models.py:51
 *   then for each GRU layer l (models.py:56-63), both directions adjacent (forward first):
 *   8+4l w_ih [2][3H, I_l]   9+4l w_hh [2][3H, H]   10+4l b_ih [2][3H]   11+4l b_hh [2][3H]
 *   then fc0_w [64, 2H], fc0_b [64], fc3_w [nc, 64], fc3_b [nc]  models.py:66-71
 * offsets/sizes are in floats.  Returns the number of segments (or < 0). */
#define MMS_MAX_SEGMENTS 64
int mms_cnngru_param_layout(const mms_cnngru_desc* d, int64_t* offsets_host, int64_t* sizes_host,
                            int32_t max_segments, int64_t* total_floats_host);

/* Frozen segments (desc.frozen_segments, the torch idiom module.requires_grad_(False)).  A segment whose bit is set is
 * never written by mms_cnngru_backward, mms_cnngru_backward_phase or mms_cnngru_train_step (its gradient slots keep
 * whatever they held; the train step's zero_grad clears only the other segments), and the backward stops as early as
 * the mask allows:
 *   - head weight gradients run only if a head segment trains;
 *   - GRU layer l's weight-gradient products run only if one of its four segments trains; its recurrence backward and
 *     the input-gradient product that feeds it only if a segment at or below layer l trains (or dx is requested);
 *   - the encoder's stage 2 (BN2/pool backward, conv2) runs only if one of segments 0-7 trains, stage 1 only if one of
 *     segments 0-4 does, the ChannelAttention gradients only if segment 0 or 1 does.
 * Empty segments (the attention weights at C < 4) and the attention segments of an attention = 0 model never keep the
 * chain alive.  Under data parallelism a phase with nothing left to do launches nothing; the SyncBN backward vectors of
 * mms_cnngru_sync_offsets are then meaningless: [3] (BN2 reductions) when segments 0-7 are all frozen, [2] (BN1
 * reductions) when segments 0-4 are.  With every bit clear nothing changes, launch for launch.
 * mms_cnngru_train_step with frozen segments needs the Adam range table (desc.adam_steps, adam_ranges_host), and no
 * range may touch a frozen segment. */
#define MMS_MAX_ADAM_RANGES 96

/* BatchNorm buffers: bn_buffers = [running_mean1[16] | running_var1[16] | running_mean2[O] |
 * running_var2[O]] float32, num_batches_tracked = int64[2] (state_dict entries
 * cnn_encoder.{1,5}.running_mean/.running_var/.num_batches_tracked). */

int64_t mms_cnngru_workspace_bytes(const mms_cnngru_desc* d);

/* models.py:73-81 forward.  x [B,C,T] -> logits [B,nc].  In training mode the workspace keeps
 * every activation the backward needs and the BN running statistics are updated. */
int mms_cnngru_forward(const mms_cnngru_desc* d, const float* x, const float* params,
                       float* bn_buffers, int64_t* num_batches_tracked, void* workspace,
                       float* logits, mms_stream_t stream);

/* trainer.py:148 loss.backward() from dlogits [B,nc]: adds every parameter gradient into
 * grads (same flat layout as params; the caller zeroes it, trainer.py:144 zero_grad).
 * dx may be NULL (inputs do not require grad in the reference, trainer.py:140). */
int mms_cnngru_backward(const mms_cnngru_desc* d, const float* x, const float* params,
                        const float* bn_buffers, void* workspace, const float* dlogits,
                        float* grads, float* dx, mms_stream_t stream);

/* Input gradient only (attribution): after mms_cnngru_forward with training = 0 and need_grad = 1 on the same workspace,
 * dx [B,C,T] = d(sum_b,c dlogits[b,c] logits[b,c]) / dx.  No parameter gradient is formed: no weight-gradient product,
 * conv or head weight gradient or side-stream work is launched, and everything runs on `stream`.  In eval mode BatchNorm
 * uses the running statistics, so the rows of the batch are independent.  Any other training / need_grad combination
 * is MMS_E_INVALID. */
int mms_cnngru_input_gradient(const mms_cnngru_desc* d, const float* x, const float* params,
                              const float* bn_buffers, void* workspace, const float* dlogits,
                              float* dx, mms_stream_t stream);

/* Integrated gradients over B windows of n = C*T samples with `steps` midpoint-rule steps, alpha_k = (k + 1/2) / steps.
 * Interpolation row r = b * steps + k.  x0 is the baseline: [B,C,T] with x0_per_window = 1, or one [C,T] shared by every
 * window with x0_per_window = 0.  A chunk is the rows [row0, row0 + nrows).
 * mms_ig_interpolate: z [nrows,C,T] = x0 + alpha_k (x - x0) and dlogits [nrows,num_classes] = one_hot(target[b]).
 * mms_ig_accumulate : A [B,C,T] += (x - x0) * dx / steps and S [B,C] (float64) += its sum over t, for dx [nrows,C,T] the
 *                     input gradient of the chunk.  Each element sums over k in increasing order, so A does not depend on
 *                     how the rows are chunked (chunks must be accumulated in row order; S to float64 rounding). */
int mms_ig_interpolate(const float* x, const float* x0, int32_t x0_per_window, const int64_t* target, int32_t B,
                       int32_t C, int32_t T, int32_t num_classes, int32_t steps, int64_t row0, int32_t nrows, float* z,
                       float* dlogits, mms_stream_t stream);
int mms_ig_accumulate(const float* x, const float* x0, int32_t x0_per_window, const float* dx, int32_t B, int32_t C,
                      int32_t T, int32_t steps, int64_t row0, int32_t nrows, float* A, double* S, mms_stream_t stream);

/* Monte-Carlo dropout (uncertainty.py): BatchNorm on its running statistics, dropout on, `samples` forward samples per
 * window.  Sample s of window b, b the window's index within the whole call of the caller, is sample row
 * r = b * samples + s, and each sample row draws the multipliers a training-mode forward of the expanded batch would draw
 * at row r: GRU site l (0 <= l < layers - 1) id = l * 2^40 + (r * L + t) * 2H + j, head site id = 2^38 + r * 64 + i, with
 * one (rng_seed, rng_offset) for every row (oracle/dropout_stream.py).
 * mms_cnngru_mc_forward: d->batch = the windows x [batch,C,T] of this chunk, d->training = 0, d->need_grad = 0 (other
 *   descriptor states, global_batch, class_weight and frozen segments are MMS_E_INVALID).  row0 = the chunk's first sample
 *   row, a multiple of `samples`.  logits [batch*samples, num_classes] in sample-row order.  The encoder and GRU layer 0
 *   run once per window (no dropout acts before layer 0's output); the layers above and the head run per sample row.  The
 *   BatchNorm buffers are read, never written.  A call whose site-0 ids would reach the head site,
 *   (row0 + batch*samples) * L * 2H >= 2^38, is MMS_E_INVALID.
 * mms_cnngru_mc_workspace_bytes: workspace of such a chunk (-1 for an invalid descriptor).
 * mms_mc_accumulate: for the rows [row0, row0 + nrows) of B*samples sample rows, logits the chunk's [nrows, num_classes],
 *   adds in float64 and in increasing s the softmax p_s to psum [B,num_classes] and -sum p_s log p_s to hsum [B] (both
 *   zeroed by the caller); a window's last sample writes probs = psum/samples, entropy = H(probs) and
 *   mutual_info = entropy - hsum/samples (float64 [B,num_classes], [B], [B]).  Chunks accumulated in row order give the
 *   same result however the rows are chunked. */
int64_t mms_cnngru_mc_workspace_bytes(const mms_cnngru_desc* d, int32_t samples);
int mms_cnngru_mc_forward(const mms_cnngru_desc* d, const float* x, const float* params, const float* bn_buffers,
                          void* workspace, int32_t samples, int64_t row0, float* logits, mms_stream_t stream);
int mms_mc_accumulate(const float* logits, int32_t B, int32_t nc, int32_t samples, int64_t row0, int32_t nrows,
                      double* psum, double* hsum, double* probs, double* entropy, double* mutual_info,
                      mms_stream_t stream);

/* Data-parallel form of the two calls above (SURVEY §8e: intra-fold DP).  `phases` is a bit mask:
 *   forward : 1 = gate + conv1 (+BN1 sums) | 2 = BN1/pool1 + conv2 (+BN2 sums) | 4 = the rest
 *   backward: 1 = head..GRU..stage-2 pool/ReLU backward (+BN2 reductions) | 2 = stage-2 BN apply, conv2
 *             gradients, stage-1 pool/ReLU backward (+BN1 reductions) | 4 = the rest
 * Between the phases the caller sum-all-reduces the float64 vectors whose byte offsets inside the
 * workspace mms_cnngru_sync_offsets() reports: [0] BN1 sums, [1] BN2 sums (forward), [2] BN1
 * reductions, [3] BN2 reductions (backward); counts are in doubles.  desc.global_batch must be set.
 * With desc.class_weight set, vector [1] has 2*cnn_out + 1 doubles: the caller writes the local sum_b w[y_b] into the last
 * one (mms_class_weight_sum) after forward phase 1 and before the exchange, and the weighted cross entropy reads the sum
 * from there (mms_cross_entropy_weighted's norm_dev).  Without class weights offsets and counts are unchanged. */
int mms_cnngru_forward_phase(const mms_cnngru_desc* d, int32_t phases, const float* x, const float* params,
                             float* bn_buffers, int64_t* num_batches_tracked, void* workspace, float* logits,
                             mms_stream_t stream);
int mms_cnngru_backward_phase(const mms_cnngru_desc* d, int32_t phases, const float* x, const float* params,
                              const float* bn_buffers, void* workspace, const float* dlogits, float* grads,
                              mms_stream_t stream);
int mms_cnngru_sync_offsets(const mms_cnngru_desc* d, int64_t* byte_offsets_host, int64_t* counts_host);
/* Cross entropy of a rank's share of a global batch: loss_out = sum_local(...)/global_batch (the per-rank
 * values add up to the global mean), dlogits = (softmax - onehot)/global_batch. */
int mms_cross_entropy_partial(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes,
                              int32_t global_batch, float* loss_out, float* dlogits, double* loss_sum_accum,
                              mms_stream_t stream);

/* The two exchange steps of intra-fold data parallelism (SURVEY §8e) WITHOUT a communication library on the data path:
 * the peers' buffers (symmetric memory mapped into this process, e.g. torch.distributed._symmetric_memory) are read
 * directly over NVLink and the ranks synchronise through flags in each other's signal pads.
 *   bufs_host / grads_host : HOST array of `world` device pointers, entry p = rank p's copy of the buffer;
 *   signals_host           : HOST array of `world` device pointers to the ranks' signal pads (uint32 words, zero at start);
 *                            a call uses words [signal_base, signal_base + 2*world) of every pad;
 *   epoch_dev              : local uint32 counter (zero at start), advanced by the call.
 * Every rank must make the same sequence of calls.  Nothing here blocks the host.
 * mms_peer_allreduce_f64: in-place sum of `count` (<= 256) doubles -- the SyncBN (sum, sum of squares) / (sum dy, sum dy*xhat)
 * vectors whose workspace offsets mms_cnngru_sync_offsets() reports.
 * mms_peer_allreduce_adam: flat gradient all-reduce FUSED with mms_adam_flat_step (trainer.py:148-149): the gradients of
 * all ranks are summed on the fly in rank order (bit-identical parameters on every rank) and consumed by the Adam update;
 * scratch2_dev: two zero-initialised local uint32.
 * Every wait inside these kernels is bounded (MMS_PEER_TIMEOUT_MS, default 2000): if a peer never signals -- a rank died,
 * made a different number of steps, or raised between two phases -- the kernel gives up, finishes with a meaningless sum and
 * counts the event.  mms_peer_status() returns that count for the current device and clears it (it synchronises the device);
 * a caller checks it wherever it reads results back.  The reference has no counterpart (its training is single-device,
 * trainer.py:57-58); this is the failure detection of the data-parallel extension (BASELINE.json configs[4]). */
int mms_peer_status(uint32_t* timeouts_host);
int mms_peer_allreduce_f64(const void* const* bufs_host, void* const* signals_host, int32_t world, int32_t rank,
                           int32_t signal_base, int32_t count, uint32_t* epoch_dev, mms_stream_t stream);
int mms_peer_allreduce_adam(float* params, const void* const* grads_host, void* const* signals_host, int32_t world,
                            int32_t rank, int32_t signal_base, float* exp_avg, float* exp_avg_sq, int64_t n,
                            const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                            int64_t* step_dev, uint32_t* epoch_dev, uint32_t* scratch2_dev, mms_stream_t stream);
/* The same with the update of mms_adam_ranges_step: only the elements inside the ranges are summed over the ranks and
 * updated; the others are neither read nor written. */
int mms_peer_allreduce_adam_ranges(float* params, const void* const* grads_host, void* const* signals_host, int32_t world,
                                   int32_t rank, int32_t signal_base, float* exp_avg, float* exp_avg_sq,
                                   const int64_t* ranges_host, int32_t nranges, int64_t* steps_dev, const float* lr_dev,
                                   float beta1, float beta2, float eps, float weight_decay, int64_t* step_dev,
                                   uint32_t* epoch_dev, uint32_t* scratch2_dev, mms_stream_t stream);

/* Gradient-norm clipping on the peer path.  mms_peer_grad_norm runs behind this rank's "gradient complete" signal: it
 * forms the norm of the world's summed gradient, each element summed in rank order with the fp32 additions of
 * mms_peer_allreduce_adam, so every rank obtains the same norm and coefficient with no further message (record and
 * clip_scratch as for mms_grad_norm; ranges_host NULL: elements [0, n)).  It uses words [signal_base, signal_base + world)
 * of every pad and its own epoch counter norm_epoch_dev (local uint32, zero at start): neither may be shared with the Adam
 * call that follows, which must read the same clip_scratch.  It has no closing barrier: the following Adam call's closing
 * barrier also tells every rank that the peers have finished this kernel.  Waits are bounded and counted as for the other
 * peer kernels.
 * mms_peer_allreduce_adam_clip / _ranges_clip: mms_peer_allreduce_adam / _ranges on coef_dev[0] * the summed gradient
 * (coef_dev = (float*)clip_scratch + 1). */
int mms_peer_grad_norm(const void* const* grads_host, void* const* signals_host, int32_t world, int32_t rank,
                       int32_t signal_base, int64_t n, const int64_t* ranges_host, int32_t nranges, const float* max_norm,
                       double* record, void* clip_scratch, uint32_t* norm_epoch_dev, mms_stream_t stream);
int mms_peer_allreduce_adam_clip(float* params, const void* const* grads_host, void* const* signals_host, int32_t world,
                                 int32_t rank, int32_t signal_base, float* exp_avg, float* exp_avg_sq, int64_t n,
                                 const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                                 int64_t* step_dev, uint32_t* epoch_dev, uint32_t* scratch2_dev, const float* coef_dev,
                                 mms_stream_t stream);
int mms_peer_allreduce_adam_ranges_clip(float* params, const void* const* grads_host, void* const* signals_host,
                                        int32_t world, int32_t rank, int32_t signal_base, float* exp_avg, float* exp_avg_sq,
                                        const int64_t* ranges_host, int32_t nranges, int64_t* steps_dev,
                                        const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                                        int64_t* step_dev, uint32_t* epoch_dev, uint32_t* scratch2_dev,
                                        const float* coef_dev, mms_stream_t stream);

/* trainer.py:69,147 CrossEntropyLoss() (mean): loss_out[0] = mean_b(lse - logit[y]),
 * dlogits = (softmax - onehot)/B (NULL to skip).  If loss_sum_accum != NULL it receives
 * += loss * B in float64 (trainer.py:152 accumulates loss.item()*batch_size on the host;
 * this keeps the sum on the device so that a step needs no sync). */
int mms_cross_entropy(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes,
                      float* loss_out, float* dlogits, double* loss_sum_accum, mms_stream_t stream);
/* CrossEntropyLoss(weight=class_weight) (mean reduction), the same kernel as the two calls above:
 * loss_out[0] = sum_b w[y_b] (lse_b - logit[b, y_b]) / W, dlogits = w[y_b] (softmax - onehot) / W, where W = *norm_dev
 * (float64; a rank's share of a data-parallel batch passes the summed slot of mms_cnngru_sync_offsets, and the per-rank
 * losses then add up to the global weighted mean) or, with norm_dev == NULL, sum_b w[y_b] over this batch.  Labels
 * outside [0, num_classes) make the loss NaN and add no gradient; W == 0 gives NaN, as torch does.  loss_sum_accum
 * receives += loss * batch.  class_weight == NULL (then norm_dev must be NULL too) is mms_cross_entropy. */
int mms_cross_entropy_weighted(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes,
                               const float* class_weight, const double* norm_dev, float* loss_out, float* dlogits,
                               double* loss_sum_accum, mms_stream_t stream);
/* out[0] = sum_b class_weight[labels[b]] over the labels in [0, num_classes) (float64, written, fixed order): the local
 * normaliser of the weighted cross entropy. */
int mms_class_weight_sum(const int64_t* labels, int32_t batch, int32_t num_classes, const float* class_weight,
                         double* out, mms_stream_t stream);

/* trainer.py:68,149 torch.optim.Adam (coupled L2 weight decay) over the flat buffer.
 * step_dev holds the number of steps already taken; the kernel uses step_dev+1 for the bias
 * corrections and increments it.  lr_dev is a device scalar (ReduceLROnPlateau writes it,
 * trainer.py:72-77,160).  scratch_dev: one int32, zero-initialised. */
int mms_adam_flat_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                       int64_t n, const float* lr_dev, float beta1, float beta2, float eps,
                       float weight_decay, int64_t* step_dev, int32_t* scratch_dev, mms_stream_t stream);
/* torch.optim.Adam over some tensors of the flat buffer, each with its own step count (torch's state['step'] is per
 * parameter; a tensor without a gradient is skipped and keeps its moments and count).  ranges_host: HOST int64
 * [nranges][3] = (offset, count, slot) in floats, disjoint, nranges in [0, MMS_MAX_ADAM_RANGES]; range k uses
 * steps_dev[slot] + 1 for its bias corrections and increments it.  Elements outside every range are neither read nor
 * written.  step_dev still advances by one per call (the fused step's dropout stream offset reads it).  The arithmetic
 * of every element is mms_adam_flat_step's. */
int mms_adam_ranges_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, const int64_t* ranges_host,
                         int32_t nranges, int64_t* steps_dev, const float* lr_dev, float beta1, float beta2, float eps,
                         float weight_decay, int64_t* step_dev, int32_t* scratch_dev, mms_stream_t stream);

/* Gradient-norm clipping, torch.nn.utils.clip_grad_norm_(params, max_norm) with norm_type 2 and error_if_nonfinite=False,
 * between the backward and Adam:
 *   total_norm = || the gradient of the trainable elements ||_2,  coef = clamp(max_norm / (total_norm + 1e-6), max = 1),
 *   and Adam (coupled weight decay) runs on coef * g.
 * The sum of squares is formed in float64 in a fixed order and rounded once to the fp32 total_norm, so the norm is
 * bit-reproducible (it differs from torch's per-tensor fp32 norms in the last bits).  For a given fp32 total_norm the
 * coefficient is torch's bit for bit: reciprocal(total_norm + 1e-6f) * max_norm, a NaN kept by the clamp; a non-finite norm
 * therefore makes the parameters NaN, as in torch.  The gradient buffer keeps the UNCLIPPED gradient.
 * clip_scratch (MMS_GRAD_CLIP_SCRATCH_BYTES, zero-initialised, one per concurrently running step): float32 [0] = the last
 * step's total norm, [1] = its coefficient; the rest is the kernels' own.
 * record (float64 [5], may be NULL; the caller zeroes it, e.g. per epoch) accumulates: [0] the sum of the finite norms,
 * [1] their maximum, [2] the steps with coef < 1, [3] the steps with a non-finite norm, [4] the steps.
 * mms_grad_norm: the norm over the ranges of ranges_host ((offset, count, slot) rows as for mms_adam_ranges_step; the slots
 *   are ignored) or, with ranges_host == NULL, over grads[0, n).  One launch; max_norm is a device float32 scalar.
 * mms_adam_flat_clip_step / mms_adam_ranges_clip_step: mms_adam_flat_step / mms_adam_ranges_step on coef_dev[0] * g
 *   (coef_dev = (float*)clip_scratch + 1 after mms_grad_norm).  With coef 1 the result is theirs bit for bit. */
#define MMS_GRAD_CLIP_SCRATCH_BYTES 1040
int mms_grad_norm(const float* grads, int64_t n, const int64_t* ranges_host, int32_t nranges, const float* max_norm,
                  double* record, void* clip_scratch, mms_stream_t stream);
int mms_adam_flat_clip_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                            int64_t n, const float* lr_dev, float beta1, float beta2, float eps,
                            float weight_decay, int64_t* step_dev, int32_t* scratch_dev, const float* coef_dev,
                            mms_stream_t stream);
int mms_adam_ranges_clip_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                              const int64_t* ranges_host, int32_t nranges, int64_t* steps_dev, const float* lr_dev,
                              float beta1, float beta2, float eps, float weight_decay, int64_t* step_dev,
                              int32_t* scratch_dev, const float* coef_dev, mms_stream_t stream);

/* trainer.py:130,140-142 -- one batch of DataLoader(dataset, batch_size, shuffle=True) (main.py:111) assembled on
 * the device: out_x[b, :] = data[perm[cursor + b], :], out_y[b] = labels[perm[cursor + b]] for b < batch.
 * data: float32 [n_rows, row_floats] (the normalised [N, C*W] window array), labels int64 [n_rows], perm: int64
 * permutation (NULL = identity), *cursor_dev: int64 position inside perm (NULL = 0).  With advance != 0 the kernel
 * moves *cursor_dev forward by `batch` when it is done, so a captured CUDA graph (gather + train step) can be
 * replayed once per batch with no host work; scratch_dev: one zero-initialised int32. */
int mms_batch_gather(const float* data, const int64_t* labels, const int64_t* perm, int64_t* cursor_dev,
                     int64_t n_rows, int64_t row_floats, int32_t batch, float* out_x, int64_t* out_y,
                     int32_t advance, int32_t* scratch_dev, mms_stream_t stream);

/* trainer.py:217-228 -- the per-batch bookkeeping of Trainer.evaluate: *loss_sum += sum_b(lse_b - logit[b, y_b])
 * (float64; the reference adds loss.item() * batch), preds_out[b] = argmax_c logits[b, c] (first maximum, as
 * torch.argmax of the softmax), confusion[y_b * nc + pred_b] += 1 (int64 [nc, nc], rows = true class).
 * accuracy_score and the weighted f1_score of trainer.py:229-230 are functions of that matrix.
 * preds_out, confusion and loss_sum may each be NULL. */
int mms_eval_accumulate(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes,
                        int64_t* preds_out, int64_t* confusion, double* loss_sum, mms_stream_t stream);
/* The same with CrossEntropyLoss(weight=class_weight): the rows are cut into groups of `group` consecutive rows (the
 * evaluation loader's batches; group <= 0: one group of `batch` rows, the last group may be shorter) and every group g of
 * n_g rows adds n_g * sum_{b in g} w[y_b] l_b / sum_{b in g} w[y_b] to *loss_sum (float64, groups in order), as the
 * reference adds loss.item() * batch per loader batch.  Predictions and confusion counts are those of
 * mms_eval_accumulate; class_weight == NULL is mms_eval_accumulate. */
int mms_eval_accumulate_weighted(const float* logits, const int64_t* labels, int32_t batch, int32_t num_classes,
                                 const float* class_weight, int32_t group, int64_t* preds_out, int64_t* confusion,
                                 double* loss_sum, mms_stream_t stream);

/* One whole training step, trainer.py:144-149: zero_grad, forward, CE, backward, Adam.
 * (With world_size > 1 the host calls forward/backward/adam separately around its NCCL
 * all-reduce instead.)  With d->clip_max_norm set, mms_grad_norm over the trainable elements (the Adam range table, or
 * every non-empty segment) runs after the backward and the clipped Adam replaces Adam: one launch more. */
int mms_cnngru_train_step(const mms_cnngru_desc* d, const float* x, const int64_t* labels,
                          float* params, float* grads, float* exp_avg, float* exp_avg_sq,
                          float* bn_buffers, int64_t* num_batches_tracked, void* workspace,
                          float* logits, float* loss_out, double* loss_sum_accum,
                          const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                          int64_t* step_dev, int32_t* scratch_dev, mms_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Operator-level entry points (the same kernels the composed calls launch), for unit parity
 * tests and for callers that use one layer on its own.
 * ---------------------------------------------------------------------------------------- */

/* models.py:24-31 ChannelAttention.forward.  hidden = C/4 may be 0 (gate == 0.5).
 * mean_out/gate_out [B,C]; y may be NULL (gate only; the model folds the gate into conv1). */
int mms_chan_attn_fwd(const float* x, const float* w1, const float* w2, int32_t B, int32_t C, int32_t T,
                      float* mean_out, float* gate_out, float* y, mms_stream_t stream);
/* Backward of the above: dy [B,C,T] -> dx [B,C,T] (may be NULL), dw1, dw2 (+=). scratch: 4*B*C floats. */
int mms_chan_attn_bwd(const float* x, const float* dy, const float* w1, const float* w2,
                      const float* mean, const float* gate, int32_t B, int32_t C, int32_t T,
                      float* dx, float* dw1, float* dw2, float* scratch, mms_stream_t stream);

/* models.py:46 / :50  Conv1d(bias=False).  which = 1: k7 s2 p3 (C_in = any <= 16, C_out 16);
 * which = 2: k5 s2 p2 (C_in 16, C_out = cnn_out).  gate [B,C_in] optional (x*gate fused).
 * stats (float64 [2][C_out]: sum, sum of squares over (B,L_out)) optional, accumulated (+=). */
int mms_conv1d_fwd(int32_t which, const float* x, const float* w, const float* gate, int32_t B,
                   int32_t c_in, int32_t c_out, int32_t l_in, float* y, double* stats, mms_stream_t stream);
/* The same convolution as an implicit GEMM on the tensor cores: TMA-staged input tile (the zero padding is TMA's
 * out-of-bounds fill), im2col + 3xTF32 operand expansion in shared memory, tcgen05.mma.kind::tf32 with the accumulator in
 * TMEM.  Same arguments and results (fp32-class accuracy); needs l_in % 4 == 0, l_in >= 64, x 16-byte aligned and
 * C_out <= 32.  mms_conv1d_fwd uses it when MMS_CONV_TC=1 (measured slower than the SIMT kernel at K = 42 / 80). */
int mms_conv1d_fwd_tc(int32_t which, const float* x, const float* w, const float* gate, int32_t B,
                      int32_t c_in, int32_t c_out, int32_t l_in, float* y, double* stats, mms_stream_t stream);
/* dgrad: dy [B,C_out,L_out] -> dx [B,C_in,L_in] (may be NULL) and, if xdot != NULL,
 * dgate[b,c] += sum_t dx[b,c,t]*xdot[b,c,t] (the only part of conv1's dgrad training needs). */
int mms_conv1d_dgrad(int32_t which, const float* dy, const float* w, int32_t B, int32_t c_in, int32_t c_out,
                     int32_t l_in, float* dx, const float* xdot, float* dgate, mms_stream_t stream);
/* wgrad: dw[o,c,k] += sum_{b,l} dy[b,o,l] * gate[b,c] * x[b,c,s*l+k-p]. */
int mms_conv1d_wgrad(int32_t which, const float* x, const float* dy, const float* gate, int32_t B,
                     int32_t c_in, int32_t c_out, int32_t l_in, float* dw, mms_stream_t stream);

/* models.py:47-49 / :51-53  BatchNorm1d + ReLU + MaxPool1d(3,2,1) fused.
 * training: batch statistics from `stats` (as produced by mms_conv1d_fwd), running buffers
 * updated (momentum 0.1, unbiased variance), nbt incremented; eval: running buffers.
 * time_major = 1 writes out[b, l, c] (models.py:77 permute(0,2,1) for free). */
int mms_bn_relu_pool_fwd(const float* y, const double* stats, const float* gamma, const float* beta,
                         float* running_mean, float* running_var, int64_t* nbt, int32_t B, int32_t C,
                         int32_t l_in, int32_t training, int32_t time_major, float* out, mms_stream_t stream);
/* Backward: dout (layout per time_major) -> dy [B,C,L_in] (in-place capable scratch), dgamma/dbeta (+=).
 * red: float64 [2][C] zero-initialised scratch. */
int mms_bn_relu_pool_bwd(const float* y, const double* stats, const float* gamma, const float* beta,
                         const float* running_mean, const float* running_var, const float* dout,
                         int32_t B, int32_t C, int32_t l_in, int32_t training, int32_t time_major,
                         float* dy, float* dgamma, float* dbeta, double* red, mms_stream_t stream);

/* GEMMs used for the GRU input projections and their gradients (models.py:78, the
 * x @ W_ih^T + b_ih part of nn.GRU):
 *   nt : C[m,n]  = sum_k A[m*lda+k] * W[n*ldw+k] + bias[n]
 *   nn : C[m,n] (+)= sum_k A[m*lda+k] * W[k*ldw+n]
 *   tn : C[i,j] += sum_m A[m*lda+acol(i)] * Bm[row(m)*ldb+j], bias_grad[i] += sum_m A[m*lda+acol(i)]
 *        acol(i) = i < a_split ? i : i + a_skip;  row(m) = m + shift within each block of
 *        `seq` rows (rows shifted outside their block read as zero) -- this is h_{t-1}. */
/* Tensor-core version of the nt form: TMA-staged operands, tcgen05.mma kind::tf32 with the 3xTF32
 * operand split (fp32-level accuracy), accumulators in TMEM.  C[m,n] (+)= sum_k A[m,k] W[n,k] + bias[n].
 * A and W must be 16-byte aligned with lda, ldw multiples of 4. */
int mms_tc_gemm_nt(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                   float* C, int64_t ldc, int32_t M, int32_t N, int32_t K, int32_t accumulate, mms_stream_t stream);
/* Tensor-core version of the tn form below (same arguments and meaning as mms_gemm_tn_acc): both row-major operands
 * are consumed MN-major by tcgen05.mma.kind::tf32 (3xTF32 split), split-K over the grid, partial tiles added to C
 * with red.global.add; the bias gradient is the product with an implicit column of ones.  Requires 16-byte aligned
 * operands, lda/ldb/ldc % 4 == 0, N1 % 32 == 0 (<= 256), N2 % 32 == 0 (<= 224, 0 = bias gradient only),
 * a_split % 32 == 0, a_skip % 32 == 0, M >= 128. */
int mms_tc_gemm_tn(const float* A, int64_t lda, int32_t a_split, int32_t a_skip, const float* Bm, int64_t ldb,
                   int32_t shift, int32_t seq, float* C, int64_t ldc, float* bias_grad,
                   int32_t M, int32_t N1, int32_t N2, mms_stream_t stream);
/* Several tensor-core TN products (2..4, each within the limits of mms_tc_gemm_tn) in ONE launch: the weight-gradient
 * products of a GRU layer (reference models.py:56-63 backward: dW_ih, dW_hh, db_ih, db_hh of both directions) reduce over
 * the same B*L rows, so one grid of ~148 CTAs covers all of them.  Used by the model when MMS_TN_BATCH=1. */
typedef struct {
    const float* A; int64_t lda; int32_t a_split, a_skip;
    const float* Bm; int64_t ldb; int32_t shift, seq;
    float* C; int64_t ldc; float* bias_grad;
    int32_t M, N1, N2;
} mms_tn_call;
int mms_tc_gemm_tn_batch(const mms_tn_call* calls_host, int32_t n, mms_stream_t stream);
int mms_gemm_nt_bias(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                     float* C, int64_t ldc, int32_t M, int32_t N, int32_t K, mms_stream_t stream);
int mms_gemm_nn(const float* A, int64_t lda, const float* W, int64_t ldw, float* C, int64_t ldc,
                int32_t M, int32_t N, int32_t K, int32_t accumulate, mms_stream_t stream);
/* Few-row products (M <= 256, K <= 256, K % 4 == 0, 16-byte aligned operands with strides that are multiples of 4): the B
 * rows of the top GRU layer's single reverse step (models.py:79 keeps only outputs[:, -1, :], SURVEY 3.2) -- its input
 * projection in the forward pass and the input gradient of that step in the backward pass.
 *   C[m,n] = sum_k a(m,k) W(n,k) (+ bias[n]);  W(n,k) = W[n*ldw + k] (w_kmajor != 0) or W[k*ldw + n]
 *   drop_mode 1: a(m,k) = A[m,k] * m(drop_base + m*drop_row_stride + k)  (models.py:62 inter-layer dropout on the operand)
 *   drop_mode 2: C[m,n] *= m(drop_base + m*drop_row_stride + n)          (the same multipliers on the gradient)
 * with the multipliers of mms_dropout_apply. */
int mms_gemm_skinny(const float* A, int64_t lda, const float* W, int64_t ldw, int32_t w_kmajor, const float* bias,
                    float* C, int64_t ldc, int32_t M, int32_t N, int32_t K, int32_t drop_mode, int64_t drop_base,
                    int64_t drop_row_stride, float dropout_p, uint64_t rng_seed, uint64_t rng_offset,
                    const int64_t* rng_offset_dev, mms_stream_t stream);
int mms_gemm_tn_acc(const float* A, int64_t lda, int32_t a_split, int32_t a_skip, const float* Bm, int64_t ldb,
                    int32_t shift, int32_t seq, float* C, int64_t ldc, float* bias_grad,
                    int32_t M, int32_t N1, int32_t N2, mms_stream_t stream);

/* models.py:62 inter-layer GRU dropout as a streaming pass: out[i] = in[i] * m(base_id + i) with
 * m in {0, 1/(1-p)} drawn from the counter-based stream (seed, offset, element id); in == out is
 * allowed.  Forward and backward call it with the same ids, so they see the same mask. */
int mms_dropout_apply(const float* in, float* out, int64_t n, int64_t base_id, float dropout_p,
                      uint64_t rng_seed, uint64_t rng_offset, const int64_t* rng_offset_dev, mms_stream_t stream);

/* The GRU recurrence of one direction (models.py:56-63; gate order r,z,n; h0 = 0).  H is 32, 64 or
 * 128.  At H = 128 every pointer and stride must be 16-byte / 4-float aligned (the shared-memory-ring
 * kernels are the only ones built for that size) and MMS_GRU_FWD_V2=0 / MMS_GRU_BWD_RING=0 are refused.
 * gi[(b*gi_bs + t*gi_ts) + 0..3H) are the input projections (incl. b_ih).  Runs `nsteps` steps
 * starting at t0 and moving by dt (+1 forward, -1 reverse).  Writes h to hs[b*hs_bs + t*hs_ts + j]
 * and, if stash != NULL, (r,z,n,W_hn h + b_hn) to
 * stash[(b*st_bs + t*st_ts) + 0..4H). */
typedef struct {
    const float* gi; int64_t gi_bs, gi_ts;
    const float* w_hh; const float* b_hh;
    float* hs; int64_t hs_bs, hs_ts;
    float* hs_drop; int64_t drop_base;   /* reserved, must be NULL / 0: use mms_dropout_apply */
    float* stash; int64_t st_bs, st_ts;
    int32_t t0, dt, nsteps;
} mms_gru_dir_fwd;
int mms_gru_recur_fwd(const mms_gru_dir_fwd* dirs_host, int32_t ndirs, int32_t B, int32_t H,
                      float dropout_p, uint64_t rng_seed, uint64_t rng_offset, const int64_t* rng_offset_dev,
                      mms_stream_t stream);

/* Reverse-time pass of one direction.  dout (optional) is the gradient w.r.t. the emitted h,
 * indexed like hs; dout_last [B, dl_ld] (optional) is added at the forward-order LAST step
 * only (or at the first one if dl_at_first); dh_head/W0 (optional): initial dh[b,k] += sum_i dh_head[b*64+i] * w0[i*w0_ld + w0_col + k].
 * drop_base / drop_mask are reserved and must be 0 (apply mms_dropout_apply to dout first).  Writes D[(b*d_bs + t*d_ts) + 0..4H) = (d r_pre, d z_pre, d n_pre, d q). */
typedef struct {
    const float* w_hh;
    const float* stash; int64_t st_bs, st_ts;
    const float* hs; int64_t hs_bs, hs_ts;
    const float* dout; int64_t do_bs, do_ts; int64_t drop_base; int32_t drop_mask;
    const float* dout_last; int64_t dl_ld; int32_t dl_at_first;  /* 1: add dout_last at the FIRST forward step instead */
    const float* dh_head; const float* w0; int64_t w0_ld; int32_t w0_col;
    float* D; int64_t d_bs, d_ts;
    int32_t t0, dt, nsteps;
} mms_gru_dir_bwd;
int mms_gru_recur_bwd(const mms_gru_dir_bwd* dirs_host, int32_t ndirs, int32_t B, int32_t H,
                      float dropout_p, uint64_t rng_seed, uint64_t rng_offset, const int64_t* rng_offset_dev,
                      mms_stream_t stream);

/* models.py:79-80 classifier head on last [B,2H]: Linear(2H,64)+ReLU+Dropout+Linear(64,nc).
 * hid_out [B,64] keeps the post-ReLU activations for the backward. */
int mms_head_fwd(const float* last, const float* w0, const float* b0, const float* w3, const float* b3,
                 int32_t B, int32_t H2, int32_t nc, float dropout_p, uint64_t rng_seed, uint64_t rng_offset,
                 const int64_t* rng_offset_dev, float* hid_out, float* logits, mms_stream_t stream);
int mms_head_bwd(const float* last, const float* hid, const float* dlogits, const float* w3,
                 int32_t B, int32_t H2, int32_t nc, float dropout_p, uint64_t rng_seed, uint64_t rng_offset,
                 const int64_t* rng_offset_dev, float* dhid, float* dw0, float* db0, float* dw3, float* db3,
                 mms_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Preprocess path (reference preprocess.py:70-75 resample_signal -> scipy.signal.resample,
 * preprocess.py:189-200 window stacking, dataset.py:37-48 normalisation).
 * ---------------------------------------------------------------------------------------- */

/* FFT resampling of `n_sig` real float64 signals of length n_in to length n_out
 * (scipy.signal.resample semantics, Fourier method, no window).  x [n_sig][n_in] ->
 * y [n_sig][n_out], both float64, rows contiguous. */
int64_t mms_resample_workspace_bytes(int64_t n_in, int64_t n_out, int32_t n_sig);
int mms_resample_f64(const double* x, int64_t n_in, int64_t n_out, int32_t n_sig, double* y,
                     void* workspace, int64_t workspace_bytes, mms_stream_t stream);

/* preprocess.py:189-200: out[w, i, c] = streams[c][starts[w] + i] for w < n_win, i < win, c < n_ch.
 * streams: HOST array of n_ch device pointers (float64 rows of length stream_len); out float64 [n_win, win, n_ch]
 * (out_f32 = 0) or float32 [n_win, n_ch, win] already permuted as dataset.py:63 does (out_f32 = 1,
 * in which case (x - shift[c]) * scale[c] is applied, log1p first where log_flag[c] != 0). */
int mms_window_gather(const double* const* streams, int32_t n_ch, int64_t stream_len,
                      const int64_t* starts, int32_t n_win, int32_t win, int32_t out_f32,
                      const double* shift, const double* scale, const int32_t* log_flag,
                      void* out, mms_stream_t stream);

/* dataset.py:37-48 statistics over the WINDOWED array without materialising it: for each
 * channel, sum and sum of squares (of log1p(x) where log_flag) over all (window, sample)
 * pairs, i.e. each stream sample weighted by the number of windows covering it.
 * sums float64 [n_ch][2], zero-initialised by the caller. */
int mms_window_stats(const double* const* streams, int32_t n_ch, int64_t stream_len,
                     const int64_t* starts, int32_t n_win, int32_t win, const int32_t* log_flag,
                     double* sums, mms_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MMS_B200_H */
