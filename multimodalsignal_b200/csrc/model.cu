// CnnGruAttentionModel (reference models.py:34-81) as a chain of hand-written kernels:
// parameter layout, workspace carving and the forward / backward / train-step launch sequences.
// Nothing here allocates or synchronises; one call enqueues the whole chain on the caller's stream
// (so a Python caller pays one ctypes call per pass and the chain can be captured in a CUDA graph).
#include "mms_common.cuh"
#include <string.h>
#include <stdlib.h>

namespace mms {

// launchers defined in the other translation units
int launch_chan_gate(const float*, const float*, const float*, int, int, int, float*, float*, cudaStream_t);
int launch_chan_param_bwd(const float*, const float*, const float*, const float*, const float*, int, int, float*, float*, float*,
                          float*, cudaStream_t);
int launch_conv_fwd(int, const float*, const float*, const float*, int, int, int, int, float*, double*, cudaStream_t);
int launch_conv_dgrad(int, const float*, const float*, int, int, int, int, float*, const float*, float*, cudaStream_t, const BnBwd* = nullptr);
int launch_conv_wgrad(int, const float*, const float*, const float*, int, int, int, int, float*, cudaStream_t, const BnBwd* = nullptr);
int launch_bn_relu_pool_fwd(const float*, const double*, const float*, const float*, float*, float*, int64_t*, int, int, int, int,
                            int, float*, cudaStream_t, int Bstat);
int launch_bn_relu_pool_bwd(const float*, const double*, const float*, const float*, const float*, const float*, const float*, int,
                            int, int, int, int, float*, float*, float*, double*, cudaStream_t, int which, int Bstat, float grad_scale);
int launch_gemm_nt_bias(const float*, int64_t, const float*, int64_t, const float*, float*, int64_t, int, int, int, cudaStream_t);
int launch_gemm_nn(const float*, int64_t, const float*, int64_t, float*, int64_t, int, int, int, int, cudaStream_t);
bool gemm_skinny_supported(const float*, int64_t, const float*, int64_t, int, int, int, int);
int launch_gemm_skinny(const float*, int64_t, const float*, int64_t, int, const float*, float*, int64_t, int, int, int, int, int64_t, int64_t,
                       float, uint64_t, uint64_t, const int64_t*, cudaStream_t);
int launch_gemm_tn_acc(const float*, int64_t, int, int, const float*, int64_t, int, int, float*, int64_t, float*, int, int, int,
                       cudaStream_t);
bool tc_gemm_tn_supported(const float*, int64_t, int, int, const float*, int64_t, float*, int64_t, int, int, int);
int launch_tc_gemm_tn(const float*, int64_t, int, int, const float*, int64_t, int, int, float*, int64_t, float*, int, int, int,
                      cudaStream_t);
int launch_gru_fwd(const mms_gru_dir_fwd*, int, int, int, float, uint64_t, uint64_t, const int64_t*, cudaStream_t);
int launch_gru_bwd(const mms_gru_dir_bwd*, int, int, int, float, uint64_t, uint64_t, const int64_t*, cudaStream_t);
int launch_head_fwd2(const float*, int64_t, const float*, int64_t, int, const float*, const float*, const float*, const float*, int,
                     int, int, float, uint64_t, uint64_t, const int64_t*, float*, float*, float*, cudaStream_t, int64_t);
int launch_head_bwd(const float*, const float*, const float*, const float*, int, int, int, float, uint64_t, uint64_t,
                    const int64_t*, float*, float*, float*, float*, float*, cudaStream_t);
int launch_cross_entropy(const float*, const int64_t*, int, int, float*, float*, double*, cudaStream_t, int div_batch,
                         const float* class_weight, const double* norm);
int launch_head_ce_fused(const float*, int64_t, const float*, int64_t, int, const float*, const float*, const float*, const float*,
                         const int64_t*, int, int, int, float, uint64_t, uint64_t, const int64_t*, int, float*, float*, float*, float*,
                         float*, float*, int32_t*, float*, double*, cudaStream_t, const float* class_weight);
int launch_adam(float*, const float*, float*, float*, int64_t, const float*, float, float, float, float, int64_t*, int32_t*,
                cudaStream_t);
int launch_adam_ranges(float*, const float*, float*, float*, const AdamRanges&, int64_t*, const float*, float, float, float, float,
                       int64_t*, int32_t*, cudaStream_t);
int launch_grad_norm(const float*, const AdamRanges&, const float*, double*, void*, cudaStream_t);
int launch_adam_clip(float*, const float*, float*, float*, int64_t, const float*, float, float, float, float, int64_t*, int32_t*,
                     const float*, cudaStream_t);
int launch_adam_ranges_clip(float*, const float*, float*, float*, const AdamRanges&, int64_t*, const float*, float, float, float,
                            float, int64_t*, int32_t*, const float*, cudaStream_t);
int launch_chan_dx(const float*, const float*, const float*, int, int, int, float*, cudaStream_t);
bool conv_fused_supported(const float*, int, int, int);
bool conv_bwd_supported(const float*, int, int, int);
int64_t conv2_bwd_scratch_floats(int, int);
int64_t conv1_bwd_scratch_floats(int, int);
int conv2_bwd_parts(int, int);
int launch_pool_bwd_tm(const float*, const double*, const float*, const float*, const float*, const float*, const float*, int, int, int,
                       int, float*, double*, cudaStream_t, int);
int launch_pool_bwd_ncl(const float*, const double*, const float*, const float*, const float*, const float*, const float*, int, int, int,
                        int, float*, double*, cudaStream_t, int);
int launch_conv2_bwd(const float*, const float*, const float*, int, int, float*, float*, cudaStream_t, const BnBwd*);
int launch_wgrad_reduce(const float*, int, int, float*, cudaStream_t);
int launch_conv2_w_relayout(const float*, float*, cudaStream_t);
int64_t conv2_w_relayout_floats();
int launch_conv1_bwd(const float*, const float*, const float*, const float*, const float*, const float*, const float*, int, int, int,
                     float*, int*, float*, float*, float*, cudaStream_t, const BnBwd*);
int launch_attn_conv1_fwd(const float*, const float*, const float*, const float*, int, int, int, int, float*, float*, float*, double*,
                          const float*, int, float*, float*,
                          cudaStream_t);
int launch_bn_pool_conv2_fwd(const float*, const double*, const float*, const float*, float*, float*, int64_t*, int, int, const float*,
                             int, int, int, int, float*, float*, double*, cudaStream_t);
int launch_conv2_w_relayout_fwd(const float*, int, float*, cudaStream_t);
int launch_tc_gemm_nt(const float*, int64_t, const float*, int64_t, const float*, float*, int64_t, int, int, int, int, cudaStream_t);
int launch_tc_gemm_nt_drop(const float*, int64_t, const float*, int64_t, const float*, float*, int64_t, int, int, int, int, cudaStream_t,
                           float, uint64_t, uint64_t, const int64_t*, int64_t, int);
bool tc_gemm_nt_drop_supported(const float*, int64_t, int);
bool tc_gemm_supported(const float*, int64_t, const float*, int64_t, int, int, int);
constexpr int TC_MIN_ROWS = 1024;      // below this a single tcgen05 CTA is pure latency: the SIMT kernels win
int launch_transpose_pad(const float*, int, int, float*, int64_t, int, cudaStream_t);
struct TransposeJobs {
    const float* W[4];
    float* out[4];
    int64_t ldo[4];
    int rows[4], cols[4], col_off[4], pad[4];
};
int launch_transpose_pad_multi(const TransposeJobs&, int, cudaStream_t);
int launch_dropout_apply(const float*, float*, int64_t, int64_t, float, uint64_t, uint64_t, const int64_t*, cudaStream_t);
int launch_dropout_rows(const float*, float*, int, int, int64_t, int64_t, float, uint64_t, uint64_t, const int64_t*, cudaStream_t);

constexpr int MAX_LAYERS = 8;
constexpr int64_t DROP_LAYER_STRIDE = 1ll << 40;

// MMS_DISABLE_TC=1 keeps every GEMM on the fp32 SIMT kernels (debugging / A-B measurements)
static bool use_tc() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("MMS_DISABLE_TC"); v = (e && e[0] == '1') ? 0 : 1; }
    return v == 1;
}

// MMS_BN_FOLD=0 keeps the BatchNorm-backward apply as its own pass instead of folding it into conv dgrad / wgrad (A/B)
static bool bn_fold() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("MMS_BN_FOLD"); v = (e && e[0] == '0') ? 0 : 1; }
    return v == 1;
}

// The TN kernel takes at most 256 gradient rows (N1, two UMMA M = 128 tiles) and 224 columns (N2).  At hidden size 128 the
// gradients have N1 = 3H = 384 rows, and the upper layers' W_ih gradient N2 = 2H = 256 columns: such a problem is cut into
// row halves (the a_split / a_skip column map of D moved past the rows before the cut) times column halves, and only the
// first column half adds the bias gradient.  A problem that fits -- every one at hidden size 32 and 64 -- is passed through.
constexpr int TN_PIECES_MAX = 4;
static int tn_split(const TnCall& c, TnCall* out) {
    const int n1_parts = c.N1 > 256 ? 2 : 1, n2_parts = c.N2 > 224 ? 2 : 1;
    const int n1 = c.N1 / n1_parts, n2 = c.N2 / n2_parts;
    int n = 0;
    for (int i = 0; i < n1_parts; ++i) {
        const int r0 = i * n1;                 // first gradient row of the piece: D column acol(r0)
        for (int j = 0; j < n2_parts; ++j) {
            TnCall q = c;
            q.N1 = n1;
            if (r0 < c.a_split) { q.A = c.A + r0; q.a_split = c.a_split - r0; }
            else { q.A = c.A + r0 + c.a_skip; q.a_split = n1; q.a_skip = 0; }
            q.N2 = n2;
            q.Bm = c.Bm ? c.Bm + (int64_t)j * n2 : nullptr;
            q.C = c.C ? c.C + (int64_t)r0 * c.ldc + (int64_t)j * n2 : nullptr;
            q.bias_grad = c.bias_grad && j == 0 ? c.bias_grad + r0 : nullptr;
            out[n++] = q;
        }
    }
    return n;
}

static bool tn_tc_ok(const TnCall& c) {
    return tc_gemm_tn_supported(c.A, c.lda, c.a_split, c.a_skip, c.N2 > 0 ? c.Bm : nullptr, c.ldb, c.N2 > 0 ? c.C : nullptr, c.ldc,
                                c.M, c.N1, c.N2);
}

// Weight-gradient (TN) products: tcgen05 split-K kernel when the shape allows it (after tn_split), fp32 SIMT otherwise.
static int gemm_tn(const float* A, int64_t lda, int a_split, int a_skip, const float* Bm, int64_t ldb, int shift, int seq, float* C,
                   int64_t ldc, float* bias_grad, int M, int N1, int N2, cudaStream_t st) {
    if (use_tc() && M >= 1024) {
        TnCall piece[TN_PIECES_MAX];
        const int np = tn_split({A, lda, a_split, a_skip, Bm, ldb, shift, seq, C, ldc, bias_grad, M, N1, N2}, piece);
        bool ok = true;
        for (int j = 0; j < np; ++j) ok = ok && tn_tc_ok(piece[j]);
        for (int j = 0; ok && j < np; ++j) {
            const TnCall& c = piece[j];
            const int rc = launch_tc_gemm_tn(c.A, c.lda, c.a_split, c.a_skip, c.Bm, c.ldb, c.shift, c.seq, c.C, c.ldc, c.bias_grad, c.M,
                                             c.N1, c.N2, st);
            if (rc) return rc;
        }
        if (ok) return MMS_OK;
    }
    return launch_gemm_tn_acc(A, lda, a_split, a_skip, Bm, ldb, shift, seq, C, ldc, bias_grad, M, N1, N2, st);
}

int launch_tc_gemm_tn_batch(const TnCall*, int, cudaStream_t);

// Several TN products on one stream: one launch of the batched tensor-core kernel when MMS_TN_BATCH=1 (experiment) and every
// problem qualifies for it, otherwise one launch each (the default).
static int gemm_tn_group(const TnCall* c, int n, cudaStream_t st) {
    bool batch = n > 1 && n <= 4 && use_tc() && option_get("TN_BATCH", 1) == 1;
    for (int j = 0; batch && j < n; ++j)
        batch = c[j].M >= 1024 && c[j].N1 > 0 &&
                tc_gemm_tn_supported(c[j].A, c[j].lda, c[j].a_split, c[j].a_skip, c[j].N2 > 0 ? c[j].Bm : nullptr, c[j].ldb,
                                     c[j].N2 > 0 ? c[j].C : nullptr, c[j].ldc, c[j].M, c[j].N1, c[j].N2);
    if (batch) return launch_tc_gemm_tn_batch(c, n, st);
    for (int j = 0; j < n; ++j) {
        int rc = gemm_tn(c[j].A, c[j].lda, c[j].a_split, c[j].a_skip, c[j].Bm, c[j].ldb, c[j].shift, c[j].seq, c[j].C, c[j].ldc,
                         c[j].bias_grad, c[j].M, c[j].N1, c[j].N2, st);
        if (rc) return rc;
    }
    return MMS_OK;
}

// Up to four TN products on one stream, cut to the TN kernel's limits (tn_split; at hidden size 32 / 64 nothing is cut) and run in
// groups of four.
static int gemm_tn_many(const TnCall* c, int n, cudaStream_t st) {
    constexpr int MAX_CALLS = 4;
    MMS_REQUIRE(n >= 1 && n <= MAX_CALLS, "gemm_tn_many: 1..%d problems", MAX_CALLS);
    TnCall pieces[MAX_CALLS * TN_PIECES_MAX];
    int np = 0;
    for (int j = 0; j < n; ++j) {
        if (use_tc() && c[j].M >= 1024) np += tn_split(c[j], pieces + np);
        else pieces[np++] = c[j];
    }
    for (int j0 = 0; j0 < np; j0 += 4) {
        const int rc = gemm_tn_group(pieces + j0, np - j0 < 4 ? np - j0 : 4, st);
        if (rc) return rc;
    }
    return MMS_OK;
}

// Side streams: weight-gradient kernels do not feed the backward critical path (recurrence -> dx ->
// recurrence -> conv chain), so they are forked onto two library-owned streams and joined before the
// caller's next kernel (Adam).  Event fork/join works identically in eager mode and under CUDA-graph
// capture (the side streams become branches of the captured graph).  MMS_DISABLE_STREAMS=1 serialises.
struct SideStreams {
    cudaStream_t s[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t fork_ev[16] = {}, join_ev[3] = {}, aux_ev = nullptr;
    bool ok = false;
};
static int g_streams_disabled = -1;
static SideStreams* side_streams() {
    static SideStreams per_dev[16];
    if (g_streams_disabled < 0) { const char* e = getenv("MMS_DISABLE_STREAMS"); g_streams_disabled = (e && e[0] == '1') ? 1 : 0; }
    if (g_streams_disabled) return nullptr;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
    SideStreams& ss = per_dev[dev];
    if (!ss.ok) {
        for (int i = 0; i < 3; ++i)
            if (cudaStreamCreateWithFlags(&ss.s[i], cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        for (int i = 0; i < 16; ++i)
            if (cudaEventCreateWithFlags(&ss.fork_ev[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
        for (int i = 0; i < 3; ++i)
            if (cudaEventCreateWithFlags(&ss.join_ev[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&ss.aux_ev, cudaEventDisableTiming) != cudaSuccess) return nullptr;
        ss.ok = true;
    }
    return &ss;
}
struct Forker {
    SideStreams* ss;
    cudaStream_t main;
    int n_forks = 0;
    bool used[3] = {false, false, false};
    Forker(cudaStream_t m) : ss(side_streams()), main(m) {}
    // stream on which work that only depends on what `main` has enqueued so far may run
    cudaStream_t fork(int which) {
        if (!ss || n_forks >= 16) return main;
        if (cudaEventRecord(ss->fork_ev[n_forks], main) != cudaSuccess) return main;
        if (cudaStreamWaitEvent(ss->s[which], ss->fork_ev[n_forks], 0) != cudaSuccess) return main;
        ++n_forks;
        used[which] = true;
        return ss->s[which];
    }
    // one early result of a side stream that `main` needs before that stream's final join: mark() after the producer has been
    // enqueued on side stream `which`, wait_mark() in front of the consumer on `main`
    bool marked = false;
    int mark(int which) {
        if (!ss || !used[which]) return MMS_OK;       // the producer ran on `main` itself
        MMS_CUDA(cudaEventRecord(ss->aux_ev, ss->s[which]));
        marked = true;
        return MMS_OK;
    }
    int wait_mark() {
        if (!marked) return MMS_OK;
        MMS_CUDA(cudaStreamWaitEvent(main, ss->aux_ev, 0));
        marked = false;
        return MMS_OK;
    }
    int join_one(int i) {
        if (!ss || !used[i]) return MMS_OK;
        MMS_CUDA(cudaEventRecord(ss->join_ev[i], ss->s[i]));
        MMS_CUDA(cudaStreamWaitEvent(main, ss->join_ev[i], 0));
        used[i] = false;
        return MMS_OK;
    }
    int join() {
        for (int i = 0; i < 3; ++i) {
            int rc = join_one(i);
            if (rc) return rc;
        }
        return MMS_OK;
    }
};

// C[m,n] = sum_k A[m,k] W[n,k] + bias[n]: tcgen05 (3xTF32) when the operands qualify, fp32 SIMT otherwise
static int gemm_nt(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, float* C, int64_t ldc, int M, int N,
                   int K, cudaStream_t st) {
    if (use_tc() && M >= TC_MIN_ROWS && tc_gemm_supported(A, lda, W, ldw, M, N, K))
        return launch_tc_gemm_nt(A, lda, W, ldw, bias, C, ldc, M, N, K, 0, st);
    return launch_gemm_nt_bias(A, lda, W, ldw, bias, C, ldc, M, N, K, st);
}

struct Dims {
    int B, Bg, C, T, nc, O, H, layers, A;      // Bg: global batch (== B unless data-parallel)
    int L1c, P1, L2c, L;   // conv1 out, pool1 out, conv2 out, pool2 out (= GRU sequence length)
    bool training, attention, need_grad, drop_gru, drop_head;
    bool weighted;         // desc.class_weight set: one more float64 (the normaliser sum_b w[y_b]) after the BN2 sums
    float p;
};

static int make_dims(const mms_cnngru_desc* d, Dims* o) {
    MMS_REQUIRE(d, "null descriptor");
    o->B = d->batch; o->C = d->in_channels; o->T = d->seq_len; o->nc = d->num_classes; o->O = d->cnn_out;
    o->H = d->hidden; o->layers = d->layers; o->A = d->in_channels / 4;
    MMS_REQUIRE(o->B >= 1, "batch must be >= 1 (got %d)", o->B);
    o->Bg = d->global_batch > 0 ? d->global_batch : o->B;
    MMS_REQUIRE(o->Bg >= o->B, "global_batch %d smaller than the local batch %d", o->Bg, o->B);
    MMS_REQUIRE(o->C >= 1 && o->C <= 16, "in_channels %d outside [1,16]", o->C);
    MMS_REQUIRE(o->nc >= 1 && o->nc <= 8, "num_classes %d outside [1,8]", o->nc);
    MMS_REQUIRE(o->O == 16 || o->O == 32 || o->O == 64, "cnn_out_channels %d not in {16,32,64}", o->O);
    MMS_REQUIRE(o->H == 32 || o->H == 64 || o->H == 128, "gru_hidden_size %d not in {32,64,128}", o->H);
    MMS_REQUIRE(o->layers >= 1 && o->layers <= MAX_LAYERS, "gru_num_layers %d outside [1,%d]", o->layers, MAX_LAYERS);
    o->L1c = conv_out_len(o->T, CONV1_K, CONV1_S, CONV1_P);
    MMS_REQUIRE(o->T >= 1 && o->L1c >= 1, "seq_len %d too short", o->T);
    // the BatchNorm / pool kernels stage whole rows (T / 2 floats) in shared memory and the fused encoder kernels take at most
    // 32 position tiles per row: windows beyond 16384 samples (60 s at > 273 Hz) are refused here, not at some launch
    MMS_REQUIRE(o->T <= 16384, "seq_len %d: windows longer than 16384 samples are not supported", o->T);
    o->P1 = pool_out_len(o->L1c);
    o->L2c = conv_out_len(o->P1, CONV2_K, CONV2_S, CONV2_P);
    MMS_REQUIRE(o->L2c >= 1, "seq_len %d too short", o->T);
    o->L = pool_out_len(o->L2c);
    o->training = d->training != 0;
    o->attention = d->attention != 0;
    o->need_grad = d->need_grad != 0;
    o->p = d->dropout_p;
    MMS_REQUIRE(o->p >= 0.f && o->p < 1.f, "dropout %f outside [0,1)", (double)o->p);
    o->drop_gru = o->training && o->p > 0.f && o->layers > 1;   // nn.GRU applies dropout only between layers
    o->drop_head = o->training && o->p > 0.f;
    o->weighted = d->class_weight != nullptr;
    return MMS_OK;
}

struct ParamOff {
    int64_t ca_w1, ca_w2, conv1_w, bn1_g, bn1_b, conv2_w, bn2_g, bn2_b;
    int64_t w_ih[MAX_LAYERS], w_hh[MAX_LAYERS], b_ih[MAX_LAYERS], b_hh[MAX_LAYERS];
    int64_t fc0_w, fc0_b, fc3_w, fc3_b, total;
    int nseg;
    int64_t off[MMS_MAX_SEGMENTS], size[MMS_MAX_SEGMENTS];
};

static void make_params(const Dims& m, ParamOff* p) {
    int64_t cur = 0;
    int n = 0;
    auto seg = [&](int64_t count) {
        const int64_t o = cur;
        p->off[n] = o; p->size[n] = count; ++n;
        cur = align_up(cur + count, 4);
        return o;
    };
    p->ca_w1 = seg((int64_t)m.A * m.C);
    p->ca_w2 = seg((int64_t)m.C * m.A);
    p->conv1_w = seg((int64_t)CONV1_CO * m.C * CONV1_K);
    p->bn1_g = seg(CONV1_CO);
    p->bn1_b = seg(CONV1_CO);
    p->conv2_w = seg((int64_t)m.O * CONV2_CI * CONV2_K);
    p->bn2_g = seg(m.O);
    p->bn2_b = seg(m.O);
    for (int l = 0; l < m.layers; ++l) {
        const int I = l == 0 ? m.O : 2 * m.H;
        p->w_ih[l] = seg((int64_t)2 * 3 * m.H * I);
        p->w_hh[l] = seg((int64_t)2 * 3 * m.H * m.H);
        p->b_ih[l] = seg((int64_t)2 * 3 * m.H);
        p->b_hh[l] = seg((int64_t)2 * 3 * m.H);
    }
    p->fc0_w = seg((int64_t)HEAD_HID * 2 * m.H);
    p->fc0_b = seg(HEAD_HID);
    p->fc3_w = seg((int64_t)m.nc * HEAD_HID);
    p->fc3_b = seg(m.nc);
    p->total = cur;
    p->nseg = n;
}

// Which parts of the backward pass run, from desc.frozen_segments (include/mms_b200.h, "Frozen segments").  A segment
// trains when its bit is clear and it has elements; the attention segments of an attention = 0 model never train.
struct Live {
    bool seg[MMS_MAX_SEGMENTS];      // the segment's gradient is written
    bool head_w;                     // a head segment trains
    bool layer_w[MAX_LAYERS];        // one of GRU layer l's four segments trains
    bool recur[MAX_LAYERS];          // layer l's recurrence backward runs: a segment at or below it trains, or dx is wanted
    bool enc2, enc1, attn;           // encoder stage 2 (segments 0-7), stage 1 (0-4), ChannelAttention (0-1)
};

static Live liveness(const Dims& m, const ParamOff& po, uint64_t frozen, bool want_dx) {
    Live v;
    for (int s = 0; s < MMS_MAX_SEGMENTS; ++s)
        v.seg[s] = s < po.nseg && po.size[s] > 0 && !((frozen >> s) & 1ull) && (s >= 2 || m.attention);
    auto any = [&](int lo, int hi) { bool a = false; for (int s = lo; s <= hi; ++s) a = a || v.seg[s]; return a; };
    v.attn = any(0, 1);
    v.enc1 = any(0, 4) || want_dx;
    v.enc2 = v.enc1 || any(5, 7);
    v.head_w = any(8 + 4 * m.layers, 11 + 4 * m.layers);
    bool below = v.enc2;
    for (int l = 0; l < m.layers; ++l) {
        v.layer_w[l] = any(8 + 4 * l, 11 + 4 * l);
        below = below || v.layer_w[l];
        v.recur[l] = below;
    }
    return v;
}

// zero_grad of the trainable segments: one memset per run of segments without a frozen bit (the whole buffer when nothing is
// frozen), so that frozen gradient slots keep their contents
static int zero_trainable(float* G, const ParamOff& po, uint64_t frozen, cudaStream_t st) {
    int s = 0;
    while (s < po.nseg) {
        if ((frozen >> s) & 1ull) { ++s; continue; }
        int e = s;
        while (e + 1 < po.nseg && !((frozen >> (e + 1)) & 1ull)) ++e;
        const int64_t lo = po.off[s], hi = e + 1 < po.nseg ? po.off[e + 1] : po.total;
        MMS_CUDA(cudaMemsetAsync(G + lo, 0, (size_t)(hi - lo) * sizeof(float), st));
        s = e + 1;
    }
    return MMS_OK;
}

struct Workspace {
    // zeroed at the start of every forward
    double* stats1; double* stats2;
    // zeroed at the start of every backward
    double* red1; double* red2; float* dgate; int* row_counter;
    size_t fwd_zero_bytes, bwd_zero_bytes;
    char* fwd_zero; char* bwd_zero;
    float *mean, *gate, *y1, *p1, *y2, *seq, *c2_wt;
    float *gi[MAX_LAYERS], *hs[MAX_LAYERS], *outd[MAX_LAYERS], *stash[MAX_LAYERS];   // bottom layers
    float *gi_tf, *gi_tr, *hs_tf, *h_tr, *stash_tf, *stash_tr, *last, *hid;
    float *wT_top, *wT[MAX_LAYERS], *dx_extra;
    int32_t* head_counter; float* rowloss;
    float *dhid, *dlogits, *D_tf, *D_tr, *D[MAX_LAYERS], *dxa, *dxb, *dy2, *dp1, *dy1, *ca_scratch, *c2_part, *c1_part, *c2_wd;
    float* gsink;          // where kernels that write several segments put the gradients of frozen ones
    int64_t total;
};

static void carve(const Dims& m, char* base, Workspace* w) {
    int64_t cur = 0;
    auto take = [&](int64_t bytes) {
        char* p = base ? base + cur : nullptr;
        cur = align_up(cur + bytes, 256);
        return p;
    };
    const int64_t B = m.B, L = m.L, H = m.H, M = B * L;
    const int64_t f = sizeof(float);
    // BN batch sums (+ with class weights the weighted loss's normaliser, summed over the ranks with the BN2 sums) + the fused
    // head's CTA counter
    const int wslot = m.weighted ? 1 : 0;
    w->fwd_zero_bytes = sizeof(double) * (2 * (CONV1_CO + m.O) + wslot) + 16;
    w->fwd_zero = take((int64_t)w->fwd_zero_bytes);
    w->stats1 = (double*)w->fwd_zero;
    w->stats2 = w->stats1 ? w->stats1 + 2 * CONV1_CO : nullptr;
    w->head_counter = w->stats1 ? (int32_t*)(w->stats2 + 2 * m.O + wslot) : nullptr;
    const int64_t bz = (int64_t)sizeof(double) * 2 * (CONV1_CO + m.O) + align_up(B * m.C, 4) * f + align_up(B, 4) * (int64_t)sizeof(int);
    w->bwd_zero = take(bz);
    w->red1 = (double*)w->bwd_zero;
    w->red2 = w->red1 ? w->red1 + 2 * CONV1_CO : nullptr;
    w->dgate = w->red1 ? (float*)(w->red2 + 2 * m.O) : nullptr;
    w->row_counter = w->red1 ? (int*)(w->dgate + align_up(B * m.C, 4)) : nullptr;     // conv1_bwd: chunks of a row that have finished
    w->bwd_zero_bytes = bz;
    w->mean = (float*)take(B * m.C * f);
    w->gate = (float*)take(B * m.C * f);
    w->y1 = (float*)take(B * CONV1_CO * m.L1c * f);
    w->p1 = (float*)take(B * CONV1_CO * m.P1 * f);
    w->y2 = (float*)take(B * m.O * m.L2c * f);
    w->seq = (float*)take(M * m.O * f);
    w->c2_wt = (float*)take((int64_t)m.O * CONV2_CI * CONV2_K * f);     // conv2 weights as [ci*5 + k][o] for the fused forward
    for (int l = 0; l < m.layers - 1; ++l) {
        w->gi[l] = (float*)take(M * 6 * H * f);
        w->hs[l] = (float*)take(M * 2 * H * f);
        w->outd[l] = m.drop_gru ? (float*)take(M * 2 * H * f) : w->hs[l];
        w->stash[l] = m.need_grad ? (float*)take(2 * M * 4 * H * f) : nullptr;
    }
    w->gi_tf = (float*)take(M * 3 * H * f);
    w->gi_tr = (float*)take(B * 3 * H * f);
    w->hs_tf = (float*)take(M * H * f);
    w->h_tr = (float*)take(B * H * f);
    w->stash_tf = m.need_grad ? (float*)take(M * 4 * H * f) : nullptr;
    w->stash_tr = m.need_grad ? (float*)take(B * 4 * H * f) : nullptr;
    w->last = (float*)take(B * 2 * H * f);
    w->hid = (float*)take(B * HEAD_HID * f);
    w->rowloss = (float*)take(B * f);
    if (m.need_grad) {
        w->dhid = (float*)take(B * HEAD_HID * f);
        w->dlogits = (float*)take(B * 8 * f);
        w->D_tf = (float*)take(M * 4 * H * f);
        w->D_tr = (float*)take(B * 4 * H * f);
        for (int l = 0; l < m.layers - 1; ++l) w->D[l] = (float*)take(M * 8 * H * f);
        const int64_t widest = 2 * H > m.O ? 2 * H : m.O;
        w->wT_top = (float*)take(2 * widest * 3 * H * f);
        for (int l = 0; l < m.layers - 1; ++l) w->wT[l] = (float*)take(widest * 8 * H * f);
        w->dx_extra = (float*)take(B * widest * f);
        w->dxa = (float*)take(M * widest * f);
        w->dxb = (float*)take(M * widest * f);
        w->dy2 = (float*)take(B * m.O * m.L2c * f);
        w->dp1 = (float*)take(B * CONV1_CO * m.P1 * f);
        w->dy1 = (float*)take(B * CONV1_CO * m.L1c * f);
        w->ca_scratch = (float*)take(4 * B * m.C * f);
        w->c2_part = (float*)take(conv2_bwd_scratch_floats(m.B, m.P1) * f);      // partial conv2 weight gradients, one per CTA
        w->c1_part = (float*)take(conv1_bwd_scratch_floats(m.B, m.C) * f);       // partial conv1 G per (row, chunk)
        w->c2_wd = (float*)take(conv2_w_relayout_floats() * f);                  // conv2 weights as [o][k][ci]
        int64_t sink = (int64_t)HEAD_HID * 2 * H;                                  // the largest segment such a kernel writes
        if ((int64_t)m.O * CONV2_CI * CONV2_K > sink) sink = (int64_t)m.O * CONV2_CI * CONV2_K;
        if ((int64_t)CONV1_CO * 16 * CONV1_K > sink) sink = (int64_t)CONV1_CO * 16 * CONV1_K;
        w->gsink = (float*)take(sink * f);
    }
    w->total = cur;
}

// phases: bit 0 = gate + conv1 (+ BN1 batch sums), bit 1 = BN1/pool1 + conv2 (+ BN2 sums), bit 2 = the rest.
// A data-parallel caller all-reduces the float64 BN sums between the phases (SyncBN); 7 = everything.
// Training-step fusion (mms_cnngru_train_step): with `fl` the head forward, CrossEntropyLoss and the head's input-side
// backward are ONE launch at the end of the forward pass (head_ce_fused_kernel); model_backward is then told that dhid /
// dlogits exist (head_done) and only computes the head's weight gradients, on a side stream.
struct FusedLoss {
    const int64_t* labels;
    float* loss_out;
    double* loss_sum_accum;
    float* grads;            // zero_grad of the fused step: cleared on a side stream of the forward (nullptr: the caller did it)
    const ParamOff* po;      // ... segment by segment: frozen segments (desc.frozen_segments) keep their slots
    uint64_t frozen;
    bool zero_bwd;           // the backward follows in the same call chain: clear its reductions with the forward's
};

// the fused forward encoder kernels run (and attn_conv1_fwd_kernel leaves the re-arranged conv2 weights in the workspace)
static bool fwd_is_fused(const Dims& m, const float* x) {
    return option_get("CONV_FUSED", 1) == 1 && conv_fused_supported(x, m.C, m.T, m.O);
}

static int model_forward(const mms_cnngru_desc* d, const float* x, const float* P, float* bn, int64_t* nbt, void* ws,
                         float* logits, cudaStream_t st, int phases = 7, const FusedLoss* fl = nullptr) {
    Dims m;
    int rc = make_dims(d, &m);
    if (rc) return rc;
    MMS_REQUIRE(x && P && bn && ws && logits, "cnngru_forward: null pointer");
    MMS_REQUIRE(!m.training || nbt, "cnngru_forward: training mode needs num_batches_tracked");
    ParamOff po;
    make_params(m, &po);
    Workspace w;
    carve(m, (char*)ws, &w);
    const int B = m.B, H = m.H, L = m.L;
    const int64_t M = (int64_t)B * L;
    float *rm1 = bn, *rv1 = bn + CONV1_CO, *rm2 = bn + 2 * CONV1_CO, *rv2 = bn + 2 * CONV1_CO + m.O;

    const float* gate = m.attention ? w.gate : nullptr;
    // fused encoder kernels (conv_fused.cu): attention + conv1 in one cluster launch, BN1/ReLU/pool + conv2 in one launch
    const bool fused = fwd_is_fused(m, x);
    if (fused) {
        if (phases & 1) {
            // one memset for the sums of this forward AND (training step in one call) the reductions / counters of the backward
            // that follows: the two regions are adjacent, and a memset node on the chain between the loss and the first
            // recurrence of the backward costs ~4 us
            size_t zb = w.fwd_zero_bytes;
            if (fl && fl->zero_bwd && m.need_grad) zb = (size_t)((w.bwd_zero + w.bwd_zero_bytes) - w.fwd_zero);
            MMS_CUDA(cudaMemsetAsync(w.fwd_zero, 0, zb, st));
            // conv2's weights in the orders bn_pool_conv2_fwd_kernel / conv2_bwd_kernel stage them are written by this launch
            // too (a few CTAs, while their tiles are in flight): no re-layout launches, no cross-stream edges on the chain
            rc = launch_attn_conv1_fwd(x, P + po.conv1_w, P + po.ca_w1, P + po.ca_w2, m.attention ? 1 : 0, B, m.C, m.T, w.mean, w.gate,
                                       w.y1, m.training ? w.stats1 : nullptr, P + po.conv2_w, m.O, w.c2_wt,
                                       m.need_grad && m.O == 32 ? w.c2_wd : nullptr, st);
            if (rc) return rc;
        }
        if (phases & 2) {
            rc = launch_bn_pool_conv2_fwd(w.y1, w.stats1, P + po.bn1_g, P + po.bn1_b, rm1, rv1, nbt, m.Bg, m.training, w.c2_wt, 1, B,
                                          m.O, m.L1c, w.p1, w.y2, m.training ? w.stats2 : nullptr, st);
            if (rc) return rc;
        }
    }
    if ((phases & 1) && !fused) {
        MMS_CUDA(cudaMemsetAsync(w.fwd_zero, 0, w.fwd_zero_bytes, st));
        if (m.attention) {
            rc = launch_chan_gate(x, P + po.ca_w1, P + po.ca_w2, B, m.C, m.T, w.mean, w.gate, st);
            if (rc) return rc;
        }
        rc = launch_conv_fwd(1, x, P + po.conv1_w, gate, B, m.C, CONV1_CO, m.T, w.y1, m.training ? w.stats1 : nullptr, st);
        if (rc) return rc;
    }
    if ((phases & 2) && !fused) {
        rc = launch_bn_relu_pool_fwd(w.y1, w.stats1, P + po.bn1_g, P + po.bn1_b, rm1, rv1, nbt, B, CONV1_CO, m.L1c, m.training, 0, w.p1, st, m.Bg);
        if (rc) return rc;
        rc = launch_conv_fwd(2, w.p1, P + po.conv2_w, nullptr, B, CONV2_CI, m.O, m.P1, w.y2, m.training ? w.stats2 : nullptr, st);
        if (rc) return rc;
    }
    if (!(phases & 4)) return MMS_OK;
    // Side work that only reads parameters (or clears what the backward writes): forked here, joined in front of the top
    // layer's recurrence, ~80 us later -- zero_grad (trainer.py:144) of the fused training step and the transposed W_ih copies
    // of the backward's tensor-core dx products.
    Forker fka(st);
    {
        const bool tc_bwd = m.need_grad && use_tc() && M >= TC_MIN_ROWS;
        if ((fl && fl->grads) || tc_bwd) {
            cudaStream_t s1 = fka.fork(1);
            if (fl && fl->grads) {
                rc = zero_trainable(fl->grads, *fl->po, fl->frozen, s1);
                if (rc) return rc;
            }
            if (tc_bwd) {
                // W_ih^T of every layer, up to four matrices per launch; the bottom layers' copies carry zero columns where the
                // D rows hold dq
                TransposeJobs jobs;
                int nj = 0;
                auto add = [&](const float* Wm, int cols, float* out, int64_t ldo, int off, int pad) -> int {
                    jobs.W[nj] = Wm; jobs.out[nj] = out; jobs.ldo[nj] = ldo; jobs.rows[nj] = 3 * H; jobs.cols[nj] = cols;
                    jobs.col_off[nj] = off; jobs.pad[nj] = pad;
                    if (++nj < 4) return MMS_OK;
                    const int r = launch_transpose_pad_multi(jobs, nj, s1);
                    nj = 0;
                    return r;
                };
                const int I_t = m.layers == 1 ? m.O : 2 * H;
                rc = add(P + po.w_ih[m.layers - 1], I_t, w.wT_top, 3 * H, 0, 0);
                if (rc) return rc;
                for (int l = 0; l < m.layers - 1; ++l) {
                    const int I_l = l == 0 ? m.O : 2 * H;
                    for (int dd = 0; dd < 2; ++dd) {
                        rc = add(P + po.w_ih[l] + (int64_t)dd * 3 * H * I_l, I_l, w.wT[l], 8 * H, dd * 4 * H, H);
                        if (rc) return rc;
                    }
                }
                if (nj) {
                    rc = launch_transpose_pad_multi(jobs, nj, s1);
                    if (rc) return rc;
                }
            }
        }
    }
    rc = launch_bn_relu_pool_fwd(w.y2, w.stats2, P + po.bn2_g, P + po.bn2_b, rm2, rv2, nbt ? nbt + 1 : nullptr, B, m.O, m.L2c,
                                 m.training, 1, w.seq, st, m.Bg);
    if (rc) return rc;

    const float* in = w.seq;
    int I = m.O;
    bool drop_on_a = false;
    for (int l = 0; l < m.layers - 1; ++l) {
        rc = gemm_nt(in, I, P + po.w_ih[l], I, P + po.b_ih[l], w.gi[l], 6 * H, (int)M, 6 * H, I, st);
        if (rc) return rc;
        mms_gru_dir_fwd dirs[2];
        for (int dd = 0; dd < 2; ++dd) {
            mms_gru_dir_fwd& g = dirs[dd];
            memset(&g, 0, sizeof(g));
            g.gi = w.gi[l] + dd * 3 * H; g.gi_bs = (int64_t)L * 6 * H; g.gi_ts = 6 * H;
            g.w_hh = P + po.w_hh[l] + (int64_t)dd * 3 * H * H;
            g.b_hh = P + po.b_hh[l] + dd * 3 * H;
            g.hs = w.hs[l] + dd * H; g.hs_bs = (int64_t)L * 2 * H; g.hs_ts = 2 * H;
            g.stash = m.need_grad ? w.stash[l] + (int64_t)dd * M * 4 * H : nullptr;
            g.st_bs = (int64_t)L * 4 * H; g.st_ts = 4 * H;
            g.t0 = dd ? L - 1 : 0; g.dt = dd ? -1 : 1; g.nsteps = L;
        }
        rc = launch_gru_fwd(dirs, 2, B, H, m.p, d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
        if (rc) return rc;
        // models.py:62: dropout on the outputs of every layer but the last.  For the layer under the top one the multipliers
        // can ride on the A operand of the top layer's input projection (tc_gemm_nt, drop_on_a): the streaming pass that
        // materialises the dropped tensor for the other consumers (the single reverse step, the weight gradients) then runs
        // on a side stream beside that product instead of in front of it (MMS_DROP_FUSED=0: the separate pass).
        drop_on_a = m.drop_gru && l == m.layers - 2 && option_get("DROP_FUSED", 1) == 1 && use_tc() && M >= TC_MIN_ROWS &&
                    tc_gemm_supported(w.hs[l], 2 * H, P + po.w_ih[l + 1], 2 * H, (int)M, 3 * H, 2 * H);
        if (m.drop_gru && !drop_on_a) {
            rc = launch_dropout_apply(w.hs[l], w.outd[l], M * 2 * H, (int64_t)l * DROP_LAYER_STRIDE, m.p, d->rng_seed,
                                      d->rng_offset, d->rng_offset_dev, st);
            if (rc) return rc;
        }
        in = w.outd[l];
        I = 2 * H;
    }
    {   // top layer: forward direction over the whole sequence, reverse direction for its first step only
        const int l = m.layers - 1;
        cudaStream_t s_side = fka.fork(0);
        // the B rows of the single reverse step: ahead of everything else on the side stream (the recurrence waits for them).
        // With the dropout riding on the big product's A operand the dropped tensor does not exist yet: the few-row kernel
        // applies the multipliers to its own operand rows.
        const float* w_rev = P + po.w_ih[l] + (int64_t)3 * H * I;
        const float* rows = (drop_on_a ? w.hs[l - 1] : in) + (int64_t)(L - 1) * I;
        if (gemm_skinny_supported(rows, (int64_t)L * I, w_rev, I, 1, B, 3 * H, I)) {
            rc = launch_gemm_skinny(rows, (int64_t)L * I, w_rev, I, 1, P + po.b_ih[l] + 3 * H, w.gi_tr, 3 * H, B, 3 * H, I, drop_on_a ? 1 : 0,
                                    (int64_t)(l - 1) * DROP_LAYER_STRIDE + (int64_t)(L - 1) * I, (int64_t)L * I, m.p, d->rng_seed,
                                    d->rng_offset, d->rng_offset_dev, s_side);
            if (rc) return rc;
            rows = nullptr;
        }
        if (drop_on_a) {
            rc = launch_dropout_apply(w.hs[l - 1], w.outd[l - 1], M * 2 * H, (int64_t)(l - 1) * DROP_LAYER_STRIDE, m.p, d->rng_seed,
                                      d->rng_offset, d->rng_offset_dev, s_side);
            if (rc) return rc;
        }
        if (rows) {
            rc = gemm_nt(in + (int64_t)(L - 1) * I, (int64_t)L * I, w_rev, I, P + po.b_ih[l] + 3 * H, w.gi_tr, 3 * H, B, 3 * H, I, s_side);
            if (rc) return rc;
        }
        if (drop_on_a)
            rc = launch_tc_gemm_nt_drop(w.hs[l - 1], I, P + po.w_ih[l], I, P + po.b_ih[l], w.gi_tf, 3 * H, (int)M, 3 * H, I, 0, st, m.p,
                                        d->rng_seed, d->rng_offset, d->rng_offset_dev, (int64_t)(l - 1) * DROP_LAYER_STRIDE, 1);
        else
            rc = gemm_nt(in, I, P + po.w_ih[l], I, P + po.b_ih[l], w.gi_tf, 3 * H, (int)M, 3 * H, I, st);
        if (rc) return rc;
        rc = fka.join();
        if (rc) return rc;
        mms_gru_dir_fwd dirs[2];
        memset(dirs, 0, sizeof(dirs));
        dirs[0].gi = w.gi_tf; dirs[0].gi_bs = (int64_t)L * 3 * H; dirs[0].gi_ts = 3 * H;
        dirs[0].w_hh = P + po.w_hh[l]; dirs[0].b_hh = P + po.b_hh[l];
        dirs[0].hs = w.hs_tf; dirs[0].hs_bs = (int64_t)L * H; dirs[0].hs_ts = H;
        dirs[0].stash = w.stash_tf; dirs[0].st_bs = (int64_t)L * 4 * H; dirs[0].st_ts = 4 * H;
        dirs[0].t0 = 0; dirs[0].dt = 1; dirs[0].nsteps = L;
        dirs[1].gi = w.gi_tr; dirs[1].gi_bs = 3 * H; dirs[1].gi_ts = 0;
        dirs[1].w_hh = P + po.w_hh[l] + (int64_t)3 * H * H; dirs[1].b_hh = P + po.b_hh[l] + 3 * H;
        dirs[1].hs = w.h_tr; dirs[1].hs_bs = H; dirs[1].hs_ts = 0;
        dirs[1].stash = w.stash_tr; dirs[1].st_bs = 4 * H; dirs[1].st_ts = 0;
        dirs[1].t0 = L - 1; dirs[1].dt = -1; dirs[1].nsteps = 1;
        rc = launch_gru_fwd(dirs, 2, B, H, 0.f, d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
        if (rc) return rc;
    }
    if (fl && m.need_grad)
        return launch_head_ce_fused(w.hs_tf + (int64_t)(L - 1) * H, (int64_t)L * H, w.h_tr, H, H, P + po.fc0_w, P + po.fc0_b,
                                    P + po.fc3_w, P + po.fc3_b, fl->labels, B, 2 * H, m.nc, m.drop_head ? m.p : 0.f, d->rng_seed,
                                    d->rng_offset, d->rng_offset_dev, m.Bg, w.last, w.hid, logits, w.dlogits, w.dhid, w.rowloss,
                                    w.head_counter, fl->loss_out, fl->loss_sum_accum, st, d->class_weight);
    return launch_head_fwd2(w.hs_tf + (int64_t)(L - 1) * H, (int64_t)L * H, w.h_tr, H, H, P + po.fc0_w, P + po.fc0_b, P + po.fc3_w,
                            P + po.fc3_b, B, 2 * H, m.nc, m.drop_head ? m.p : 0.f, d->rng_seed, d->rng_offset, d->rng_offset_dev,
                            w.last, w.hid, logits, st, 0);
}

// Appends TN product `c` to list[n] with the frozen outputs removed: no weight gradient (C == nullptr) leaves the bias gradient
// alone (N2 = 0), neither leaves nothing.  Returns the new count.
static int tn_keep(TnCall* list, int n, TnCall c) {
    if (!c.C) { c.N2 = 0; c.Bm = nullptr; c.ldb = 0; c.ldc = 0; }
    if (!c.C && !c.bias_grad) return n;
    list[n] = c;
    return n + 1;
}

// phases: bit 0 = head ... GRU ... pool/ReLU backward of stage 2 (+ its BN reductions), bit 1 = BN apply of stage 2,
// conv2 gradients, pool/ReLU backward of stage 1 (+ reductions), bit 2 = the rest.  A data-parallel caller
// all-reduces the float64 reductions between the phases; 7 = everything.
static int model_backward(const mms_cnngru_desc* d, const float* x, const float* P, const float* bn, void* ws,
                          const float* dlogits, float* G, float* dx, cudaStream_t st, int phases = 7, bool head_done = false,
                          bool bwd_zeroed = false) {
    Dims m;
    int rc = make_dims(d, &m);
    if (rc) return rc;
    MMS_REQUIRE(m.need_grad, "cnngru_backward: the forward pass was run with need_grad = 0");
    MMS_REQUIRE(x && P && bn && ws && dlogits && G, "cnngru_backward: null pointer");
    ParamOff po;
    make_params(m, &po);
    Workspace w;
    carve(m, (char*)ws, &w);
    const int B = m.B, H = m.H, L = m.L;
    const int M = B * L;
    const float *rm1 = bn, *rv1 = bn + CONV1_CO, *rm2 = bn + 2 * CONV1_CO, *rv2 = bn + 2 * CONV1_CO + m.O;
    const float p = m.p;

    const float gscale = (float)m.B / (float)m.Bg;       // share of the global BN affine gradient this rank adds
    // conv_bwd.cu (the default when the shapes allow it): T % 32 == 0, C_out == 32, BatchNorm backward folded, no input gradient
    const bool bwd2 = bn_fold() && !dx && option_get("CONV_BWD", 1) == 1 && conv_bwd_supported(x, m.C, m.T, m.O);
    // frozen segments: what runs (Live), and the gradient slot of segment s -- nullptr where it must stay untouched (the TN
    // products and BnBwd skip null outputs), or a scratch sink for kernels that write several segments in one launch
    const Live lv = liveness(m, po, d->frozen_segments, dx != nullptr);
    auto gs = [&](int s) -> float* { return lv.seg[s] ? G + po.off[s] : nullptr; };
    auto gk = [&](int s) -> float* { return lv.seg[s] ? G + po.off[s] : w.gsink; };
    const int top = m.layers - 1;
    const int hs0 = 8 + 4 * m.layers;                    // first head segment
    Forker fk(st);
    if ((phases & 1) && (lv.head_w || lv.recur[top])) {
    if (!bwd_zeroed && lv.enc2) MMS_CUDA(cudaMemsetAsync(w.bwd_zero, 0, w.bwd_zero_bytes, st));
    const bool tc_bwd = use_tc() && M >= TC_MIN_ROWS;      // W_ih^T for the tensor-core dx products: made by the forward pass
    // conv2's weights in conv2_bwd_kernel's order: left in the workspace by the fused forward (attn_conv1_fwd_kernel); after a
    // per-layer forward they are made here, on a side stream, long before they are needed
    if (bwd2 && phases == 7 && lv.enc2 && !fwd_is_fused(m, x)) {
        rc = launch_conv2_w_relayout(P + po.conv2_w, w.c2_wd, fk.fork(1));
        if (rc) return rc;
        rc = fk.mark(1);
        if (rc) return rc;
    }
    // head: dhid feeds the top recurrence; with the fused forward it already exists and only the weight gradients remain,
    // which nothing on the chain needs -> side stream
    const bool need_dhid = !head_done && lv.recur[top];
    if (lv.head_w || need_dhid) {
        rc = launch_head_bwd(w.last, w.hid, dlogits, P + po.fc3_w, B, 2 * H, m.nc, m.drop_head ? p : 0.f, d->rng_seed, d->rng_offset,
                             d->rng_offset_dev, need_dhid ? w.dhid : nullptr, gk(hs0), gk(hs0 + 1), gk(hs0 + 2), gk(hs0 + 3),
                             head_done ? fk.fork(2) : st);
        if (rc) return rc;
    }
    if (!lv.recur[top]) return fk.join();      // head only: nothing below it trains

    const float* in_top = top == 0 ? w.seq : w.outd[top - 1];
    const int I_top = top == 0 ? m.O : 2 * H;
    float* dxcur = w.dxa;
    float* dxnext = w.dxb;
    int drop_done_for = -1;        // layer whose output-dropout gradient has already been applied by a GEMM epilogue
    // Weight gradients of the top layer: side stream 0, forked from wherever this is called.  MMS_WGRAD_DEFER=1 (experiment)
    // forks them after the NEXT layer's recurrence has been enqueued instead of right after the top one, so that they overlap
    // the conv backward chain rather than the layer-0 recurrence (whose CTAs lose issue slots to co-resident GEMM CTAs).
    auto top_wgrad = [&]() -> int {
        if (!lv.layer_w[top]) return MMS_OK;
        const int sg = 8 + 4 * top;
        float *g_wih = gs(sg), *g_whh = gs(sg + 1), *g_bih = gs(sg + 2), *g_bhh = gs(sg + 3);
        TnCall big[2];
        const int nb = tn_keep(big, 0, {w.D_tf, 4 * H, 3 * H, 0, in_top, I_top, 0, L, g_wih, I_top, g_bih, M, 3 * H, I_top});
        const int nbig = tn_keep(big, nb, {w.D_tf, 4 * H, 2 * H, H, w.hs_tf, H, -1, L, g_whh, H, g_bhh, M, 3 * H, H});
        if (nbig) {
            const int r = gemm_tn_many(big, nbig, fk.fork(0));
            if (r) return r;
        }
        // the B-row products of the single reverse step: their own side stream, beside the big products instead of behind them
        TnCall rev[2];
        int nrev = tn_keep(rev, 0, {w.D_tr, 4 * H, 3 * H, 0, in_top + (int64_t)(L - 1) * I_top, (int64_t)L * I_top, 0, 1,
                                    g_wih ? g_wih + (int64_t)3 * H * I_top : nullptr, I_top, g_bih ? g_bih + 3 * H : nullptr, B, 3 * H, I_top});
        // h_prev = 0 for the single reverse step: dW_hh(reverse) = 0, only the bias gradient remains
        nrev = tn_keep(rev, nrev, {w.D_tr, 4 * H, 2 * H, H, nullptr, 0, 0, 1, nullptr, 0, g_bhh ? g_bhh + 3 * H : nullptr, B, 3 * H, 0});
        cudaStream_t ss = nrev ? fk.fork(2) : st;
        for (int j = 0; j < nrev; ++j) {
            const TnCall& c = rev[j];
            const int r = gemm_tn(c.A, c.lda, c.a_split, c.a_skip, c.Bm, c.ldb, c.shift, c.seq, c.C, c.ldc, c.bias_grad, c.M, c.N1, c.N2, ss);
            if (r) return r;
        }
        return MMS_OK;
    };
    // MMS_WGRAD_DEFER: 0 = right behind the top recurrence (beside the dx product), 1 (default) = behind the next recurrence,
    // 2 (experiment) = behind the dx product, i.e. beside the next recurrence only
    const int defer_mode = top >= 1 && lv.recur[top - 1] ? option_get("WGRAD_DEFER", 1) : 0;
    const bool dx_top = top >= 1 ? lv.recur[top - 1] : lv.enc2;     // the top layer's input gradient is consumed
    const bool defer_top_wgrad = defer_mode >= 1;
    {
        mms_gru_dir_bwd dirs[2];
        memset(dirs, 0, sizeof(dirs));
        dirs[0].w_hh = P + po.w_hh[top];
        dirs[0].stash = w.stash_tf; dirs[0].st_bs = (int64_t)L * 4 * H; dirs[0].st_ts = 4 * H;
        dirs[0].hs = w.hs_tf; dirs[0].hs_bs = (int64_t)L * H; dirs[0].hs_ts = H;
        dirs[0].dh_head = w.dhid; dirs[0].w0 = P + po.fc0_w; dirs[0].w0_ld = 2 * H; dirs[0].w0_col = 0;
        dirs[0].D = w.D_tf; dirs[0].d_bs = (int64_t)L * 4 * H; dirs[0].d_ts = 4 * H;
        dirs[0].t0 = 0; dirs[0].dt = 1; dirs[0].nsteps = L;
        dirs[1].w_hh = P + po.w_hh[top] + (int64_t)3 * H * H;
        dirs[1].stash = w.stash_tr; dirs[1].st_bs = 4 * H; dirs[1].st_ts = 0;
        dirs[1].hs = w.h_tr; dirs[1].hs_bs = H; dirs[1].hs_ts = 0;
        dirs[1].dh_head = w.dhid; dirs[1].w0 = P + po.fc0_w; dirs[1].w0_ld = 2 * H; dirs[1].w0_col = H;
        dirs[1].D = w.D_tr; dirs[1].d_bs = 4 * H; dirs[1].d_ts = 0;
        dirs[1].t0 = L - 1; dirs[1].dt = -1; dirs[1].nsteps = 1;
        rc = launch_gru_bwd(dirs, 2, B, H, p, d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
        if (rc) return rc;
        // weight gradients of the top layer (off the critical path -> side stream), here or after the next recurrence
        if (!defer_top_wgrad) {
            rc = top_wgrad();
            if (rc) return rc;
        }
        if (top >= 1 && dx_top) {
            // the single reverse step only touches the rows t = L-1: its B-row product goes to dx_extra on a side
            // stream, beside the big product below; the layer underneath adds it at t = L-1
            cudaStream_t sx = fk.fork(2);
            const float* w_rev = P + po.w_ih[top] + (int64_t)3 * H * I_top;
            if (gemm_skinny_supported(w.D_tr, 4 * H, w_rev, I_top, 0, B, I_top, 3 * H)) {
                // few-row kernel, the dropout gradient on its result: the next recurrence waits for these rows
                rc = launch_gemm_skinny(w.D_tr, 4 * H, w_rev, I_top, 0, nullptr, w.dx_extra, I_top, B, I_top, 3 * H, m.drop_gru ? 2 : 0,
                                        (int64_t)(top - 1) * DROP_LAYER_STRIDE + (int64_t)(L - 1) * I_top, (int64_t)L * I_top, p,
                                        d->rng_seed, d->rng_offset, d->rng_offset_dev, sx);
                if (rc) return rc;
            } else {
                rc = launch_gemm_nn(w.D_tr, 4 * H, w_rev, I_top, w.dx_extra, I_top, B, I_top, 3 * H, 0, sx);
                if (rc) return rc;
                if (m.drop_gru) {
                    rc = launch_dropout_rows(w.dx_extra, w.dx_extra, B, I_top, (int64_t)(top - 1) * DROP_LAYER_STRIDE + (int64_t)(L - 1) * I_top,
                                             (int64_t)L * I_top, p, d->rng_seed, d->rng_offset, d->rng_offset_dev, sx);
                    if (rc) return rc;
                }
            }
        }
        // gradient w.r.t. the top layer's input
        if (!dx_top) {
        } else if (tc_bwd && tc_gemm_supported(w.D_tf, 4 * H, w.wT_top, 3 * H, M, I_top, 3 * H)) {
            // tensor-core path: dx = D @ W_ih as an NT product against the transposed weights
            // the gradient through the dropout between layer top-1 and top (same multipliers as the forward) rides on this
            // product's epilogue instead of a separate pass over dxcur
            if (top >= 1 && m.drop_gru && option_get("DROP_FUSED", 1) == 1 && tc_gemm_nt_drop_supported(dxcur, I_top, I_top)) {
                rc = launch_tc_gemm_nt_drop(w.D_tf, 4 * H, w.wT_top, 3 * H, nullptr, dxcur, I_top, M, I_top, 3 * H, 0, st, p, d->rng_seed,
                                            d->rng_offset, d->rng_offset_dev, (int64_t)(top - 1) * DROP_LAYER_STRIDE, 0);
                drop_done_for = top - 1;
            } else {
                rc = launch_tc_gemm_nt(w.D_tf, 4 * H, w.wT_top, 3 * H, nullptr, dxcur, I_top, M, I_top, 3 * H, 0, st);
            }
            if (rc) return rc;
        } else {
            rc = launch_gemm_nn(w.D_tf, 4 * H, P + po.w_ih[top], I_top, dxcur, I_top, M, I_top, 3 * H, 0, st);
            if (rc) return rc;
        }
        // the single reverse step only touches the rows t = L-1 (B rows, SIMT)
        if (top == 0 && dx_top) {
            rc = launch_gemm_nn(w.D_tr, 4 * H, P + po.w_ih[top] + (int64_t)3 * H * I_top, I_top, dxcur + (int64_t)(L - 1) * I_top,
                                (int64_t)L * I_top, B, I_top, 3 * H, 1, st);
            if (rc) return rc;
        }
    }
    for (int l = top - 1; l >= 0 && lv.recur[l]; --l) {
        const float* in_l = l == 0 ? w.seq : w.outd[l - 1];
        const int I_l = l == 0 ? m.O : 2 * H;
        if (m.drop_gru && drop_done_for != l) {      // gradient through the dropout between layer l and l + 1 (same multipliers)
            rc = launch_dropout_apply(dxcur, dxcur, (int64_t)M * 2 * H, (int64_t)l * DROP_LAYER_STRIDE, p, d->rng_seed,
                                      d->rng_offset, d->rng_offset_dev, st);
            if (rc) return rc;
        }
        if (l == top - 1) {
            rc = fk.join_one(2);     // dx_extra is complete
            if (rc) return rc;
        }
        mms_gru_dir_bwd dirs[2];
        memset(dirs, 0, sizeof(dirs));
        for (int dd = 0; dd < 2; ++dd) {
            mms_gru_dir_bwd& g = dirs[dd];
            g.w_hh = P + po.w_hh[l] + (int64_t)dd * 3 * H * H;
            g.stash = w.stash[l] + (int64_t)dd * M * 4 * H; g.st_bs = (int64_t)L * 4 * H; g.st_ts = 4 * H;
            g.hs = w.hs[l] + dd * H; g.hs_bs = (int64_t)L * 2 * H; g.hs_ts = 2 * H;
            g.dout = dxcur + dd * H; g.do_bs = (int64_t)L * 2 * H; g.do_ts = 2 * H;
            if (l == top - 1) {      // the top layer's single reverse step contributes at t = L-1 only
                g.dout_last = w.dx_extra + dd * H; g.dl_ld = 2 * H;
                g.dl_at_first = dd;  // t = L-1 is the LAST forward step of direction 0 and the FIRST of direction 1
            }
            g.D = w.D[l] + dd * 4 * H; g.d_bs = (int64_t)L * 8 * H; g.d_ts = 8 * H;
            g.t0 = dd ? L - 1 : 0; g.dt = dd ? -1 : 1; g.nsteps = L;
        }
        if (defer_mode == 2 && l == top - 1) {
            rc = top_wgrad();
            if (rc) return rc;
        }
        rc = launch_gru_bwd(dirs, 2, B, H, p, d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
        if (rc) return rc;
        const bool tn_after = option_get("TN_AFTER_NT", 1) == 1;
        if (defer_mode == 1 && l == top - 1 && !tn_after) {
            rc = top_wgrad();
            if (rc) return rc;
        }
        // Weight gradients of this layer: side stream.  MMS_TN_AFTER_NT=1 (default since the GEMM CTAs were re-staffed: 1.7 % faster; it was 3 % slower with the earlier kernels) forks them AFTER the input-gradient product
        // below has been enqueued: both stream the same D rows, and started together the 148-CTA weight-gradient kernels
        // stretched the (critical-path) input-gradient product 2.4x (round-2 timeline); started behind it they overlap the
        // encoder's backward kernels instead.
        auto layer_wgrad = [&]() -> int {
            if (!lv.layer_w[l]) return MMS_OK;
            const int sg = 8 + 4 * l;
            float *g_wih = gs(sg), *g_whh = gs(sg + 1), *g_bih = gs(sg + 2), *g_bhh = gs(sg + 3);
            TnCall four[4];
            int n4 = 0;
            for (int dd = 0; dd < 2; ++dd) {
                const float* Dd = w.D[l] + dd * 4 * H;
                n4 = tn_keep(four, n4, {Dd, 8 * H, 3 * H, 0, in_l, I_l, 0, L, g_wih ? g_wih + (int64_t)dd * 3 * H * I_l : nullptr, I_l,
                                        g_bih ? g_bih + dd * 3 * H : nullptr, M, 3 * H, I_l});
                n4 = tn_keep(four, n4, {Dd, 8 * H, 2 * H, H, w.hs[l] + dd * H, 2 * H, dd ? 1 : -1, L,
                                        g_whh ? g_whh + (int64_t)dd * 3 * H * H : nullptr, H, g_bhh ? g_bhh + dd * 3 * H : nullptr, M, 3 * H, H});
            }
            return gemm_tn_many(four, n4, fk.fork(1 - (l & 1)));
        };
        if (!tn_after) {
            rc = layer_wgrad();
            if (rc) return rc;
        }
        if (!(l >= 1 ? lv.recur[l - 1] : lv.enc2)) {
            // nothing underneath needs this layer's input gradient
        } else if (tc_bwd && tc_gemm_supported(w.D[l], 8 * H, w.wT[l], 8 * H, M, I_l, 8 * H)) {
            // both directions in one NT product: K = [fwd 3H | (dq) | rev 3H | (dq)], zero weights on the dq columns
            rc = launch_tc_gemm_nt(w.D[l], 8 * H, w.wT[l], 8 * H, nullptr, dxnext, I_l, M, I_l, 8 * H, 0, st);
            if (rc) return rc;
        } else {
            for (int dd = 0; dd < 2; ++dd) {
                rc = launch_gemm_nn(w.D[l] + dd * 4 * H, 8 * H, P + po.w_ih[l] + (int64_t)dd * 3 * H * I_l, I_l, dxnext, I_l, M, I_l,
                                    3 * H, dd, st);
                if (rc) return rc;
            }
        }
        if (tn_after) {
            if (defer_mode == 1 && l == top - 1) {
                rc = top_wgrad();
                if (rc) return rc;
            }
            rc = layer_wgrad();
            if (rc) return rc;
        }
        float* t = dxcur; dxcur = dxnext; dxnext = t;
    }
    if (!lv.enc2) return fk.join();           // the encoder is frozen: the chain ends at the bottom GRU layer
    // dxcur = d(seq) [B, L, O] time-major
    if (bwd2)
        rc = launch_pool_bwd_tm(w.y2, w.stats2, P + po.bn2_g, P + po.bn2_b, rm2, rv2, dxcur, B, m.O, m.L2c, m.training, w.dy2, w.red2, st,
                                m.Bg);
    else
        rc = launch_bn_relu_pool_bwd(w.y2, w.stats2, P + po.bn2_g, P + po.bn2_b, rm2, rv2, dxcur, B, m.O, m.L2c, m.training, 1, w.dy2,
                                     gk(6), gk(7), w.red2, st, 1, m.Bg, gscale);
    if (rc) return rc;
    }   // phase bit 0
    if (!lv.enc2) return fk.join();
    // The BatchNorm-backward apply pass is folded into the consumers of dy (BnBwd, mms_common.cuh): w.dy2 / w.dy1 hold the
    // un-normalised gradients written by pool_relu_bwd, and conv dgrad / wgrad form dy while staging their tiles (after the
    // reductions in w.red2 / w.red1 are complete -- all-reduced by the caller under data parallelism).
    const bool fold = bn_fold();
    if (phases & 2) {
        if (!fold) {
            rc = launch_bn_relu_pool_bwd(w.y2, w.stats2, P + po.bn2_g, P + po.bn2_b, rm2, rv2, nullptr, B, m.O, m.L2c, m.training, 1, w.dy2,
                                         gk(6), gk(7), w.red2, st, 2, m.Bg, gscale);
            if (rc) return rc;
        }
        const BnBwd bn2w = {fold ? w.y2 : nullptr, w.stats2, P + po.bn2_g, P + po.bn2_b, rm2, rv2, w.red2, gs(6), gs(7), m.Bg, m.training, gscale};
        BnBwd bn2d = bn2w;
        bn2d.dgamma = nullptr; bn2d.dbeta = nullptr;
        if (bwd2) {
            // both gradients of conv2 from one staged tile; the per-CTA partial weight gradients are summed on a side stream
            if (phases != 7) {       // phase-split call (data parallel): the re-arranged weights are made here
                rc = launch_conv2_w_relayout(P + po.conv2_w, w.c2_wd, st);
                if (rc) return rc;
            }
            rc = fk.wait_mark();
            if (rc) return rc;
            // with stage 1 frozen the kernel forms the weight gradient alone (no dp1)
            rc = launch_conv2_bwd(w.dy2, w.c2_wd, w.p1, B, m.P1, lv.enc1 ? w.dp1 : nullptr, w.c2_part, st, &bn2w);
            if (rc) return rc;
            if (lv.seg[5]) {
                rc = launch_wgrad_reduce(w.c2_part, conv2_bwd_parts(B, m.P1), m.O * CONV2_CI * CONV2_K, gs(5), fk.fork(0));
                if (rc) return rc;
            }
            if (lv.enc1) {
                rc = launch_pool_bwd_ncl(w.y1, w.stats1, P + po.bn1_g, P + po.bn1_b, rm1, rv1, w.dp1, B, CONV1_CO, m.L1c, m.training, w.dy1,
                                         w.red1, st, m.Bg);
                if (rc) return rc;
            }
        } else {
        // the weight-gradient kernel also adds the BN2 affine gradients (BnBwd)
        if (lv.seg[5] || lv.seg[6] || lv.seg[7]) {
            rc = launch_conv_wgrad(2, w.p1, w.dy2, nullptr, B, CONV2_CI, m.O, m.P1, gk(5), fk.fork(0), &bn2w);
            if (rc) return rc;
        }
        if (lv.enc1) {
            rc = launch_conv_dgrad(2, w.dy2, P + po.conv2_w, B, CONV2_CI, m.O, m.P1, w.dp1, nullptr, nullptr, st, &bn2d);
            if (rc) return rc;
            rc = launch_bn_relu_pool_bwd(w.y1, w.stats1, P + po.bn1_g, P + po.bn1_b, rm1, rv1, w.dp1, B, CONV1_CO, m.L1c, m.training, 0,
                                         w.dy1, gk(3), gk(4), w.red1, st, 1, m.Bg, gscale);
            if (rc) return rc;
        }
        }
    }
    if (!(phases & 4) || !lv.enc1) return fk.join();
    if (bwd2) {
        // conv1 weight gradient, attention-gate gradient and the ChannelAttention parameter gradients in one launch
        const BnBwd bn1f = {w.y1, w.stats1, P + po.bn1_g, P + po.bn1_b, rm1, rv1, w.red1, gs(3), gs(4), m.Bg, m.training, gscale};
        rc = launch_conv1_bwd(x, w.dy1, P + po.conv1_w, m.attention ? w.gate : nullptr, w.mean, P + po.ca_w1, P + po.ca_w2, B, m.C, m.T,
                              w.c1_part, w.row_counter, gk(2), gk(0), gk(1), st, &bn1f);
        if (rc) return rc;
        return fk.join();
    }
    if (!fold) {
        rc = launch_bn_relu_pool_bwd(w.y1, w.stats1, P + po.bn1_g, P + po.bn1_b, rm1, rv1, nullptr, B, CONV1_CO, m.L1c, m.training, 0,
                                     w.dy1, gk(3), gk(4), w.red1, st, 2, m.Bg, gscale);
        if (rc) return rc;
    }
    const BnBwd bn1w = {fold ? w.y1 : nullptr, w.stats1, P + po.bn1_g, P + po.bn1_b, rm1, rv1, w.red1, gs(3), gs(4), m.Bg, m.training, gscale};
    BnBwd bn1d = bn1w;
    bn1d.dgamma = nullptr; bn1d.dbeta = nullptr;
    if (lv.seg[2] || lv.seg[3] || lv.seg[4]) {     // the weight-gradient kernel also adds the BN1 affine gradients
        rc = launch_conv_wgrad(1, x, w.dy1, m.attention ? w.gate : nullptr, B, m.C, CONV1_CO, m.T, gk(2), fk.fork(1), &bn1w);
        if (rc) return rc;
    }
    if (m.attention) {
        if ((m.A > 0 && lv.attn) || dx) {
            // dx (if requested) first receives d(x*gate); dgate[b,c] = sum_t d(x*gate) * x
            rc = launch_conv_dgrad(1, w.dy1, P + po.conv1_w, B, m.C, CONV1_CO, m.T, dx, x, w.dgate, st, &bn1d);
            if (rc) return rc;
            float* ds = dx && m.A > 0 ? w.ca_scratch : nullptr;
            rc = launch_chan_param_bwd(w.dgate, w.mean, w.gate, P + po.ca_w1, P + po.ca_w2, B, m.C, w.ca_scratch + (int64_t)B * m.C, ds,
                                       gk(0), gk(1), st);
            if (rc) return rc;
            if (dx) {
                rc = launch_chan_dx(dx, w.gate, ds, B, m.C, m.T, dx, st);
                if (rc) return rc;
            }
        }
    } else if (dx) {
        rc = launch_conv_dgrad(1, w.dy1, P + po.conv1_w, B, m.C, CONV1_CO, m.T, dx, nullptr, nullptr, st, &bn1d);
        if (rc) return rc;
    }
    return fk.join();       // every gradient is complete before the caller's next kernel (Adam)
}

int launch_encoder_eval_bwd(const float*, const float*, const float*, const float*, const float*, const float*, const float*,
                            const float*, const float*, int, int, int, float*, cudaStream_t);
int launch_attn_input_grad(const float*, const float*, const float*, const float*, const float*, int, int, int, float*, cudaStream_t);
int launch_head_input_grad(const float*, const float*, const float*, int, int, float*, cudaStream_t);

// dx only, after an eval-mode forward with need_grad = 1 (attribution): the head, GRU and encoder input gradients of
// model_backward without a single parameter gradient, all on the caller's stream.  The GRU recurrences and the NT input-gradient
// products are model_backward's; the head and the encoder use the eval-mode kernels of conv_eval_bwd.cu, where BatchNorm is an
// affine map and the pool / ReLU / BN backward of both stages folds into one launch with conv2's input gradient.
static int model_input_gradient(const mms_cnngru_desc* d, const float* x, const float* P, const float* bn, void* ws,
                                const float* dlogits, float* dx, cudaStream_t st) {
    Dims m;
    int rc = make_dims(d, &m);
    if (rc) return rc;
    MMS_REQUIRE(!m.training && m.need_grad, "cnngru_input_gradient: needs an eval-mode forward (training = 0, need_grad = 1)");
    MMS_REQUIRE(x && P && bn && ws && dlogits && dx, "cnngru_input_gradient: null pointer");
    ParamOff po;
    make_params(m, &po);
    Workspace w;
    carve(m, (char*)ws, &w);
    const int B = m.B, H = m.H, L = m.L;
    const int M = B * L;
    const bool tc_bwd = use_tc() && M >= TC_MIN_ROWS;      // W_ih^T for the tensor-core products: made by the forward pass

    rc = launch_head_input_grad(w.hid, dlogits, P + po.fc3_w, B, m.nc, w.dhid, st);
    if (rc) return rc;
    const int top = m.layers - 1;
    const int I_top = top == 0 ? m.O : 2 * H;
    float* dxcur = w.dxa;
    float* dxnext = w.dxb;
    {
        mms_gru_dir_bwd dirs[2];
        memset(dirs, 0, sizeof(dirs));
        dirs[0].w_hh = P + po.w_hh[top];
        dirs[0].stash = w.stash_tf; dirs[0].st_bs = (int64_t)L * 4 * H; dirs[0].st_ts = 4 * H;
        dirs[0].hs = w.hs_tf; dirs[0].hs_bs = (int64_t)L * H; dirs[0].hs_ts = H;
        dirs[0].dh_head = w.dhid; dirs[0].w0 = P + po.fc0_w; dirs[0].w0_ld = 2 * H; dirs[0].w0_col = 0;
        dirs[0].D = w.D_tf; dirs[0].d_bs = (int64_t)L * 4 * H; dirs[0].d_ts = 4 * H;
        dirs[0].t0 = 0; dirs[0].dt = 1; dirs[0].nsteps = L;
        dirs[1].w_hh = P + po.w_hh[top] + (int64_t)3 * H * H;
        dirs[1].stash = w.stash_tr; dirs[1].st_bs = 4 * H; dirs[1].st_ts = 0;
        dirs[1].hs = w.h_tr; dirs[1].hs_bs = H; dirs[1].hs_ts = 0;
        dirs[1].dh_head = w.dhid; dirs[1].w0 = P + po.fc0_w; dirs[1].w0_ld = 2 * H; dirs[1].w0_col = H;
        dirs[1].D = w.D_tr; dirs[1].d_bs = 4 * H; dirs[1].d_ts = 0;
        dirs[1].t0 = L - 1; dirs[1].dt = -1; dirs[1].nsteps = 1;
        rc = launch_gru_bwd(dirs, 2, B, H, 0.f, d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
        if (rc) return rc;
        const float* w_rev = P + po.w_ih[top] + (int64_t)3 * H * I_top;
        if (top >= 1) {      // the single reverse step's B rows, added by the layer underneath at t = L-1
            if (gemm_skinny_supported(w.D_tr, 4 * H, w_rev, I_top, 0, B, I_top, 3 * H))
                rc = launch_gemm_skinny(w.D_tr, 4 * H, w_rev, I_top, 0, nullptr, w.dx_extra, I_top, B, I_top, 3 * H, 0, 0,
                                        (int64_t)L * I_top, 0.f, d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
            else
                rc = launch_gemm_nn(w.D_tr, 4 * H, w_rev, I_top, w.dx_extra, I_top, B, I_top, 3 * H, 0, st);
            if (rc) return rc;
        }
        if (tc_bwd && tc_gemm_supported(w.D_tf, 4 * H, w.wT_top, 3 * H, M, I_top, 3 * H))
            rc = launch_tc_gemm_nt(w.D_tf, 4 * H, w.wT_top, 3 * H, nullptr, dxcur, I_top, M, I_top, 3 * H, 0, st);
        else
            rc = launch_gemm_nn(w.D_tf, 4 * H, P + po.w_ih[top], I_top, dxcur, I_top, M, I_top, 3 * H, 0, st);
        if (rc) return rc;
        if (top == 0) {
            rc = launch_gemm_nn(w.D_tr, 4 * H, w_rev, I_top, dxcur + (int64_t)(L - 1) * I_top, (int64_t)L * I_top, B, I_top, 3 * H,
                                1, st);
            if (rc) return rc;
        }
    }
    for (int l = top - 1; l >= 0; --l) {
        const int I_l = l == 0 ? m.O : 2 * H;
        mms_gru_dir_bwd dirs[2];
        memset(dirs, 0, sizeof(dirs));
        for (int dd = 0; dd < 2; ++dd) {
            mms_gru_dir_bwd& g = dirs[dd];
            g.w_hh = P + po.w_hh[l] + (int64_t)dd * 3 * H * H;
            g.stash = w.stash[l] + (int64_t)dd * M * 4 * H; g.st_bs = (int64_t)L * 4 * H; g.st_ts = 4 * H;
            g.hs = w.hs[l] + dd * H; g.hs_bs = (int64_t)L * 2 * H; g.hs_ts = 2 * H;
            g.dout = dxcur + dd * H; g.do_bs = (int64_t)L * 2 * H; g.do_ts = 2 * H;
            if (l == top - 1) { g.dout_last = w.dx_extra + dd * H; g.dl_ld = 2 * H; g.dl_at_first = dd; }
            g.D = w.D[l] + dd * 4 * H; g.d_bs = (int64_t)L * 8 * H; g.d_ts = 8 * H;
            g.t0 = dd ? L - 1 : 0; g.dt = dd ? -1 : 1; g.nsteps = L;
        }
        rc = launch_gru_bwd(dirs, 2, B, H, 0.f, d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
        if (rc) return rc;
        if (tc_bwd && tc_gemm_supported(w.D[l], 8 * H, w.wT[l], 8 * H, M, I_l, 8 * H)) {
            rc = launch_tc_gemm_nt(w.D[l], 8 * H, w.wT[l], 8 * H, nullptr, dxnext, I_l, M, I_l, 8 * H, 0, st);
            if (rc) return rc;
        } else {
            for (int dd = 0; dd < 2; ++dd) {
                rc = launch_gemm_nn(w.D[l] + dd * 4 * H, 8 * H, P + po.w_ih[l] + (int64_t)dd * 3 * H * I_l, I_l, dxnext, I_l, M, I_l,
                                    3 * H, dd, st);
                if (rc) return rc;
            }
        }
        float* t = dxcur; dxcur = dxnext; dxnext = t;
    }
    // dxcur = d(seq) [B, L, O] time-major -> dy1 [B, 16, L1c]
    rc = launch_encoder_eval_bwd(dxcur, w.y2, w.y1, P + po.conv2_w, P + po.bn1_g, P + po.bn1_b, P + po.bn2_g, P + po.bn2_b, bn, B,
                                 m.O, m.L1c, w.dy1, st);
    if (rc) return rc;
    // conv1's input gradient; with the attention gate it is the gradient of x * gate, reduced against x for dgate
    const bool gate_mlp = m.attention && m.A > 0;
    if (gate_mlp) MMS_CUDA(cudaMemsetAsync(w.dgate, 0, (size_t)B * m.C * sizeof(float), st));
    rc = launch_conv_dgrad(1, w.dy1, P + po.conv1_w, B, m.C, CONV1_CO, m.T, dx, gate_mlp ? x : nullptr, gate_mlp ? w.dgate : nullptr,
                           st);
    if (rc) return rc;
    if (m.attention) return launch_attn_input_grad(w.dgate, w.mean, w.gate, P + po.ca_w1, P + po.ca_w2, B, m.C, m.T, dx, st);
    return MMS_OK;
}

int launch_mc_expand(const float*, int64_t, int64_t, int, int64_t, float*, int64_t, float, uint64_t, uint64_t, const int64_t*,
                     cudaStream_t);

// MC dropout (mms_cnngru_mc_forward): eval-mode BatchNorm, dropout on, `samples` sample rows per window.  No dropout acts
// before GRU layer 0's output, so the encoder and layer 0 run once on the windows (model_forward's carve and kernels);
// layer 0's output is then broadcast to the sample rows with the first site's multipliers, and the layers above and the
// head run on the sample rows.  A 1-layer model shares its whole GRU and only the head's mask varies.
constexpr int64_t MC_SITE0_LIMIT = 1ll << 38;     // HEAD_DROP_BASE (head_opt.cu): site-0 ids must stay below it

struct McWorkspace {
    Workspace win;                                  // the windows: encoder, layer 0 (1 layer: the whole GRU)
    float* in0;                                     // [rows, L, 2H] layer 0's output per sample row, site 0 applied
    float *gi[MAX_LAYERS], *hs[MAX_LAYERS], *outd[MAX_LAYERS];   // middle layers 1 .. layers-2 on the sample rows
    float *gi_tf, *gi_tr, *hs_tf, *h_tr;            // top layer on the sample rows
    float *last_a, *last_b;                         // 1 layer: the windows' classifier input per sample row
    float *last, *hid;                              // head on the sample rows
    int64_t total;
};

static void mc_carve(const Dims& m, int samples, char* base, McWorkspace* w) {
    carve(m, base, &w->win);
    int64_t cur = w->win.total;
    auto take = [&](int64_t bytes) {
        float* p = base ? (float*)(base + cur) : nullptr;
        cur = align_up(cur + bytes, 256);
        return p;
    };
    const int64_t R = (int64_t)m.B * samples, L = m.L, H = m.H, M = R * L, f = sizeof(float);
    memset(w->gi, 0, sizeof(w->gi)); memset(w->hs, 0, sizeof(w->hs)); memset(w->outd, 0, sizeof(w->outd));
    w->in0 = w->gi_tf = w->gi_tr = w->hs_tf = w->h_tr = w->last_a = w->last_b = nullptr;
    if (m.layers >= 2) {
        w->in0 = take(M * 2 * H * f);
        for (int l = 1; l < m.layers - 1; ++l) {
            w->gi[l] = take(M * 6 * H * f);
            w->hs[l] = take(M * 2 * H * f);
            w->outd[l] = m.p > 0.f ? take(M * 2 * H * f) : w->hs[l];
        }
        w->gi_tf = take(M * 3 * H * f);
        w->gi_tr = take(R * 3 * H * f);
        w->hs_tf = take(M * H * f);
        w->h_tr = take(R * H * f);
    } else {
        w->last_a = take(R * H * f);
        w->last_b = take(R * H * f);
    }
    w->last = take(R * 2 * H * f);
    w->hid = take(R * HEAD_HID * f);
    w->total = cur;
}

// one bidirectional layer over all L steps of `rows` rows, eval: in [rows, L, I] -> gi [rows*L, 6H] -> hs [rows, L, 2H]
static int mc_bidir_layer(const Dims& m, const ParamOff& po, const float* P, int l, const float* in, int I, int rows, float* gi,
                          float* hs, const mms_cnngru_desc* d, cudaStream_t st) {
    const int H = m.H, L = m.L;
    const int64_t M = (int64_t)rows * L;
    int rc = gemm_nt(in, I, P + po.w_ih[l], I, P + po.b_ih[l], gi, 6 * H, (int)M, 6 * H, I, st);
    if (rc) return rc;
    mms_gru_dir_fwd dirs[2];
    memset(dirs, 0, sizeof(dirs));
    for (int dd = 0; dd < 2; ++dd) {
        mms_gru_dir_fwd& g = dirs[dd];
        g.gi = gi + dd * 3 * H; g.gi_bs = (int64_t)L * 6 * H; g.gi_ts = 6 * H;
        g.w_hh = P + po.w_hh[l] + (int64_t)dd * 3 * H * H;
        g.b_hh = P + po.b_hh[l] + dd * 3 * H;
        g.hs = hs + dd * H; g.hs_bs = (int64_t)L * 2 * H; g.hs_ts = 2 * H;
        g.st_bs = (int64_t)L * 4 * H; g.st_ts = 4 * H;
        g.t0 = dd ? L - 1 : 0; g.dt = dd ? -1 : 1; g.nsteps = L;
    }
    return launch_gru_fwd(dirs, 2, rows, H, 0.f, d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
}

// the top layer, eval: forward direction over the whole sequence, reverse direction for its first step only (model_forward's
// top-layer block without dropout, stash or side stream)
static int mc_top_layer(const Dims& m, const ParamOff& po, const float* P, const float* in, int I, int rows, float* gi_tf, float* gi_tr,
                        float* hs_tf, float* h_tr, const mms_cnngru_desc* d, cudaStream_t st) {
    const int H = m.H, L = m.L, l = m.layers - 1;
    const int64_t M = (int64_t)rows * L;
    const float* w_rev = P + po.w_ih[l] + (int64_t)3 * H * I;
    const float* rows_in = in + (int64_t)(L - 1) * I;
    int rc;
    if (gemm_skinny_supported(rows_in, (int64_t)L * I, w_rev, I, 1, rows, 3 * H, I))
        rc = launch_gemm_skinny(rows_in, (int64_t)L * I, w_rev, I, 1, P + po.b_ih[l] + 3 * H, gi_tr, 3 * H, rows, 3 * H, I, 0, 0, 0, 0.f,
                                d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
    else
        rc = gemm_nt(rows_in, (int64_t)L * I, w_rev, I, P + po.b_ih[l] + 3 * H, gi_tr, 3 * H, rows, 3 * H, I, st);
    if (rc) return rc;
    rc = gemm_nt(in, I, P + po.w_ih[l], I, P + po.b_ih[l], gi_tf, 3 * H, (int)M, 3 * H, I, st);
    if (rc) return rc;
    mms_gru_dir_fwd dirs[2];
    memset(dirs, 0, sizeof(dirs));
    dirs[0].gi = gi_tf; dirs[0].gi_bs = (int64_t)L * 3 * H; dirs[0].gi_ts = 3 * H;
    dirs[0].w_hh = P + po.w_hh[l]; dirs[0].b_hh = P + po.b_hh[l];
    dirs[0].hs = hs_tf; dirs[0].hs_bs = (int64_t)L * H; dirs[0].hs_ts = H;
    dirs[0].st_bs = (int64_t)L * 4 * H; dirs[0].st_ts = 4 * H;
    dirs[0].t0 = 0; dirs[0].dt = 1; dirs[0].nsteps = L;
    dirs[1].gi = gi_tr; dirs[1].gi_bs = 3 * H; dirs[1].gi_ts = 0;
    dirs[1].w_hh = P + po.w_hh[l] + (int64_t)3 * H * H; dirs[1].b_hh = P + po.b_hh[l] + 3 * H;
    dirs[1].hs = h_tr; dirs[1].hs_bs = H; dirs[1].hs_ts = 0;
    dirs[1].st_bs = 4 * H; dirs[1].st_ts = 0;
    dirs[1].t0 = L - 1; dirs[1].dt = -1; dirs[1].nsteps = 1;
    return launch_gru_fwd(dirs, 2, rows, H, 0.f, d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
}

static int mc_dims(const mms_cnngru_desc* d, int samples, int64_t row0, Dims* m) {
    int rc = make_dims(d, m);
    if (rc) return rc;
    MMS_REQUIRE(!m->training && !m->need_grad, "cnngru_mc_forward: needs training = 0 and need_grad = 0");
    MMS_REQUIRE(m->Bg == m->B && !m->weighted && d->frozen_segments == 0,
                "cnngru_mc_forward: global_batch, class_weight and frozen_segments are not used by MC dropout");
    MMS_REQUIRE(samples >= 1, "cnngru_mc_forward: samples %d < 1", samples);
    MMS_REQUIRE(row0 >= 0 && row0 % samples == 0, "cnngru_mc_forward: row0 %lld is not a window boundary", (long long)row0);
    const int64_t rows = (int64_t)m->B * samples;
    MMS_REQUIRE(rows * m->L < INT32_MAX, "cnngru_mc_forward: %lld sample rows x %d steps is too many for one call", (long long)rows,
                m->L);
    // the largest site-0 id, (row0 + rows) * L * 2H - 1, must stay below the head site's base
    MMS_REQUIRE(row0 < MC_SITE0_LIMIT && (row0 + rows) * ((int64_t)m->L * 2 * m->H) < MC_SITE0_LIMIT,
                "cnngru_mc_forward: sample rows up to %lld reach the head site's dropout ids (rows * L * 2H >= 2^38)",
                (long long)(row0 + rows));
    return MMS_OK;
}

static int model_mc_forward(const mms_cnngru_desc* d, const float* x, const float* P, const float* bn, void* ws, int samples,
                            int64_t row0, float* logits, cudaStream_t st) {
    Dims m;
    int rc = mc_dims(d, samples, row0, &m);
    if (rc) return rc;
    MMS_REQUIRE(x && P && bn && ws && logits, "cnngru_mc_forward: null pointer");
    ParamOff po;
    make_params(m, &po);
    McWorkspace w;
    mc_carve(m, samples, (char*)ws, &w);
    const int B = m.B, H = m.H, L = m.L, R = B * samples;
    const float p = m.p;
    float* bnw = const_cast<float*>(bn);             // eval mode: the running statistics are read, never written
    // shared prefix: encoder stages 1 and 2 (model_forward's kernels), BN2/ReLU/pool into the GRU input, layer 0
    rc = model_forward(d, x, P, bnw, nullptr, ws, logits, st, 3);
    if (rc) return rc;
    rc = launch_bn_relu_pool_fwd(w.win.y2, w.win.stats2, P + po.bn2_g, P + po.bn2_b, bnw + 2 * CONV1_CO, bnw + 2 * CONV1_CO + m.O, nullptr,
                                 B, m.O, m.L2c, 0, 1, w.win.seq, st, B);
    if (rc) return rc;
    const float *head_a, *head_b;
    int64_t lda, ldb;
    if (m.layers == 1) {
        rc = mc_top_layer(m, po, P, w.win.seq, m.O, B, w.win.gi_tf, w.win.gi_tr, w.win.hs_tf, w.win.h_tr, d, st);
        if (rc) return rc;
        rc = launch_mc_expand(w.win.hs_tf + (int64_t)(L - 1) * H, (int64_t)L * H, H, samples, R, w.last_a, 0, 0.f, 0, 0, nullptr, st);
        if (rc) return rc;
        rc = launch_mc_expand(w.win.h_tr, H, H, samples, R, w.last_b, 0, 0.f, 0, 0, nullptr, st);
        if (rc) return rc;
        head_a = w.last_a; lda = H; head_b = w.last_b; ldb = H;
    } else {
        rc = mc_bidir_layer(m, po, P, 0, w.win.seq, m.O, B, w.win.gi[0], w.win.hs[0], d, st);
        if (rc) return rc;
        // per sample row from here: site 0 on layer 0's output, broadcast from the windows
        const int64_t row_len = (int64_t)L * 2 * H;
        rc = launch_mc_expand(w.win.hs[0], row_len, row_len, samples, R, w.in0, row0 * row_len, p, d->rng_seed, d->rng_offset,
                              d->rng_offset_dev, st);
        if (rc) return rc;
        const float* in = w.in0;
        for (int l = 1; l < m.layers - 1; ++l) {
            rc = mc_bidir_layer(m, po, P, l, in, 2 * H, R, w.gi[l], w.hs[l], d, st);
            if (rc) return rc;
            if (p > 0.f) {
                rc = launch_dropout_apply(w.hs[l], w.outd[l], (int64_t)R * row_len, (int64_t)l * DROP_LAYER_STRIDE + row0 * row_len, p,
                                          d->rng_seed, d->rng_offset, d->rng_offset_dev, st);
                if (rc) return rc;
            }
            in = w.outd[l];
        }
        rc = mc_top_layer(m, po, P, in, 2 * H, R, w.gi_tf, w.gi_tr, w.hs_tf, w.h_tr, d, st);
        if (rc) return rc;
        head_a = w.hs_tf + (int64_t)(L - 1) * H; lda = (int64_t)L * H; head_b = w.h_tr; ldb = H;
    }
    return launch_head_fwd2(head_a, lda, head_b, ldb, H, P + po.fc0_w, P + po.fc0_b, P + po.fc3_w, P + po.fc3_b, R, 2 * H, m.nc, p,
                            d->rng_seed, d->rng_offset, d->rng_offset_dev, w.last, w.hid, logits, st, row0);
}

}  // namespace mms

using namespace mms;

extern "C" int64_t mms_cnngru_mc_workspace_bytes(const mms_cnngru_desc* d, int32_t samples) {
    Dims m;
    if (mc_dims(d, samples, 0, &m)) return -1;
    McWorkspace w;
    mc_carve(m, samples, nullptr, &w);
    return w.total;
}

extern "C" int mms_cnngru_mc_forward(const mms_cnngru_desc* d, const float* x, const float* params, const float* bn_buffers,
                                     void* workspace, int32_t samples, int64_t row0, float* logits, mms_stream_t stream) {
    return model_mc_forward(d, x, params, bn_buffers, workspace, samples, row0, logits, (cudaStream_t)stream);
}

extern "C" int mms_cnngru_param_layout(const mms_cnngru_desc* d, int64_t* offsets_host, int64_t* sizes_host, int32_t max_segments,
                                       int64_t* total_floats_host) {
    Dims m;
    int rc = make_dims(d, &m);
    if (rc) return rc;
    ParamOff po;
    make_params(m, &po);
    MMS_REQUIRE(po.nseg <= max_segments, "param_layout: need room for %d segments", po.nseg);
    for (int i = 0; i < po.nseg; ++i) {
        if (offsets_host) offsets_host[i] = po.off[i];
        if (sizes_host) sizes_host[i] = po.size[i];
    }
    if (total_floats_host) *total_floats_host = po.total;
    return po.nseg;
}

extern "C" int mms_set_side_streams(int32_t on) {
    g_streams_disabled = on ? 0 : 1;
    return MMS_OK;
}

extern "C" int64_t mms_cnngru_workspace_bytes(const mms_cnngru_desc* d) {
    Dims m;
    if (make_dims(d, &m)) return -1;
    Workspace w;
    carve(m, nullptr, &w);
    return w.total;
}

extern "C" int mms_cnngru_forward(const mms_cnngru_desc* d, const float* x, const float* params, float* bn_buffers,
                                  int64_t* num_batches_tracked, void* workspace, float* logits, mms_stream_t stream) {
    return model_forward(d, x, params, bn_buffers, num_batches_tracked, workspace, logits, (cudaStream_t)stream);
}

extern "C" int mms_cnngru_backward(const mms_cnngru_desc* d, const float* x, const float* params, const float* bn_buffers,
                                   void* workspace, const float* dlogits, float* grads, float* dx, mms_stream_t stream) {
    return model_backward(d, x, params, bn_buffers, workspace, dlogits, grads, dx, (cudaStream_t)stream);
}

extern "C" int mms_cnngru_input_gradient(const mms_cnngru_desc* d, const float* x, const float* params, const float* bn_buffers,
                                         void* workspace, const float* dlogits, float* dx, mms_stream_t stream) {
    return model_input_gradient(d, x, params, bn_buffers, workspace, dlogits, dx, (cudaStream_t)stream);
}

extern "C" int mms_cnngru_forward_phase(const mms_cnngru_desc* d, int32_t phases, const float* x, const float* params,
                                        float* bn_buffers, int64_t* num_batches_tracked, void* workspace, float* logits,
                                        mms_stream_t stream) {
    MMS_REQUIRE(phases >= 1 && phases <= 7, "forward_phase: phases must be a mask in [1,7]");
    return model_forward(d, x, params, bn_buffers, num_batches_tracked, workspace, logits, (cudaStream_t)stream, phases);
}

extern "C" int mms_cnngru_backward_phase(const mms_cnngru_desc* d, int32_t phases, const float* x, const float* params,
                                         const float* bn_buffers, void* workspace, const float* dlogits, float* grads,
                                         mms_stream_t stream) {
    MMS_REQUIRE(phases >= 1 && phases <= 7, "backward_phase: phases must be a mask in [1,7]");
    return model_backward(d, x, params, bn_buffers, workspace, dlogits, grads, nullptr, (cudaStream_t)stream, phases);
}

extern "C" int mms_cnngru_sync_offsets(const mms_cnngru_desc* d, int64_t* byte_offsets_host, int64_t* counts_host) {
    Dims m;
    int rc = make_dims(d, &m);
    if (rc) return rc;
    MMS_REQUIRE(byte_offsets_host && counts_host, "sync_offsets: null pointer");
    Workspace w;
    char* base = reinterpret_cast<char*>(4096);          // any non-null base: only differences are used
    carve(m, base, &w);
    byte_offsets_host[0] = (char*)w.stats1 - base; counts_host[0] = 2 * CONV1_CO;
    byte_offsets_host[1] = (char*)w.stats2 - base; counts_host[1] = 2 * m.O + (m.weighted ? 1 : 0);   // + sum_b w[y_b]
    byte_offsets_host[2] = (char*)w.red1 - base;   counts_host[2] = 2 * CONV1_CO;
    byte_offsets_host[3] = (char*)w.red2 - base;   counts_host[3] = 2 * m.O;
    return MMS_OK;
}

extern "C" int mms_cnngru_train_step(const mms_cnngru_desc* d, const float* x, const int64_t* labels, float* params, float* grads,
                                     float* exp_avg, float* exp_avg_sq, float* bn_buffers, int64_t* num_batches_tracked,
                                     void* workspace, float* logits, float* loss_out, double* loss_sum_accum, const float* lr_dev,
                                     float beta1, float beta2, float eps, float weight_decay, int64_t* step_dev,
                                     int32_t* scratch_dev, mms_stream_t stream) {
    cudaStream_t st = (cudaStream_t)stream;
    Dims m;
    int rc = make_dims(d, &m);
    if (rc) return rc;
    MMS_REQUIRE(m.training && m.need_grad, "train_step: descriptor must have training = need_grad = 1");
    MMS_REQUIRE(labels && grads && exp_avg && exp_avg_sq && loss_out && lr_dev && step_dev && scratch_dev, "train_step: null pointer");
    // the weighted loss is normalised by sum_b w[y_b] of THIS batch; a rank's share of a larger batch needs the global sum
    // (mms_cnngru_sync_offsets + mms_cross_entropy_weighted)
    MMS_REQUIRE(!m.weighted || m.Bg == m.B, "train_step: class weights with global_batch %d > batch %d", m.Bg, m.B);
    ParamOff po;
    make_params(m, &po);
    Workspace w;
    carve(m, (char*)workspace, &w);
    // fine-tuning: Adam over the trainable tensors' ranges, which must leave the frozen segments' (untouched) gradient slots alone
    const uint64_t frozen = d->frozen_segments;
    AdamRanges ranges;
    const bool by_range = d->adam_steps != nullptr;
    MMS_REQUIRE(by_range || (d->adam_nranges == 0 && !d->adam_ranges_host), "train_step: an Adam range table without adam_steps");
    MMS_REQUIRE(by_range || !frozen, "train_step: frozen segments need the Adam range table (adam_steps, adam_ranges_host)");
    if (by_range) {
        rc = adam_ranges_from_host(d->adam_ranges_host, d->adam_nranges, po.total, &ranges);
        if (rc) return rc;
        for (int k = 0; k < ranges.n; ++k)
            for (int sg = 0; sg < po.nseg; ++sg)
                MMS_REQUIRE(!((frozen >> sg) & 1ull) || ranges.off[k] + ranges.cnt[k] <= po.off[sg] ||
                                po.off[sg] + po.size[sg] <= ranges.off[k],
                            "train_step: Adam range %d overlaps frozen segment %d", k, sg);
    }
    const bool fuse_head = option_get("HEAD_FUSED", 1) == 1;
    // zero_grad (trainer.py:144): nothing writes a gradient before the backward pass, so with the fused head the memset runs on
    // a side stream of the forward instead of in front of its first kernel
    if (!fuse_head) {
        rc = zero_trainable(grads, po, frozen, st);
        if (rc) return rc;
    }
    const bool zero_bwd = fuse_head && fwd_is_fused(m, x);
    const FusedLoss fl = {labels, loss_out, loss_sum_accum, grads, &po, frozen, zero_bwd};
    rc = model_forward(d, x, params, bn_buffers, num_batches_tracked, workspace, logits, st, 7, fuse_head ? &fl : nullptr);  // trainer.py:146-147
    if (rc) return rc;
    if (!fuse_head) {
        rc = launch_cross_entropy(logits, labels, m.B, m.nc, loss_out, w.dlogits, loss_sum_accum, st, m.Bg, d->class_weight,
                                  nullptr);                                                                // trainer.py:147
        if (rc) return rc;
    }
    rc = model_backward(d, x, params, bn_buffers, workspace, w.dlogits, grads, nullptr, st, 7, fuse_head, zero_bwd);        // trainer.py:148
    if (rc) return rc;
    if (d->clip_max_norm) {
        // clip_grad_norm_ over the trainable elements: the Adam ranges, or every non-empty segment (never the padding between them)
        AdamRanges nr;
        if (by_range) {
            nr = ranges;
        } else {
            nr.n = 0;
            for (int sg = 0; sg < po.nseg; ++sg)
                if (po.size[sg] > 0) {
                    nr.off[nr.n] = po.off[sg]; nr.cnt[nr.n] = po.size[sg]; nr.slot[nr.n] = 0;
                    ++nr.n;
                }
        }
        rc = launch_grad_norm(grads, nr, d->clip_max_norm, d->clip_record, d->clip_scratch, st);
        if (rc) return rc;
        const float* coef = reinterpret_cast<const float*>(d->clip_scratch) + 1;
        if (by_range)
            return launch_adam_ranges_clip(params, grads, exp_avg, exp_avg_sq, ranges, d->adam_steps, lr_dev, beta1, beta2, eps,
                                           weight_decay, step_dev, scratch_dev, coef, st);
        return launch_adam_clip(params, grads, exp_avg, exp_avg_sq, po.total, lr_dev, beta1, beta2, eps, weight_decay, step_dev,
                                scratch_dev, coef, st);
    }
    if (by_range)
        return launch_adam_ranges(params, grads, exp_avg, exp_avg_sq, ranges, d->adam_steps, lr_dev, beta1, beta2, eps, weight_decay,
                                  step_dev, scratch_dev, st);
    return launch_adam(params, grads, exp_avg, exp_avg_sq, po.total, lr_dev, beta1, beta2, eps, weight_decay, step_dev,
                       scratch_dev, st);                                                          // trainer.py:149
}
