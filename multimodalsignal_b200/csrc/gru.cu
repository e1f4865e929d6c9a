// GRU recurrence (reference models.py:56-63 nn.GRU; PyTorch gate order r,z,n; h0 = 0), forward and
// reverse-time backward, as persistent kernels: one CTA owns R batch rows of one direction for the
// whole sequence, so there is no inter-CTA communication and one block barrier per time step.
//
// The kernels are latency-bound: a 240-step serial chain whose every step is a 3H x H mat-vec plus
// the gate non-linearities.  The design therefore minimises the per-step dependent chain and the
// instruction count, not bytes:
//   * a CTA has 2*H threads; thread (p, q) = (tid >> 2, tid & 3) owns TWO hidden units (p and p + H/2)
//     and a quarter q of the reduction index.  Its 3 gates x H/4 weights for both units sit in
//     registers as float2 pairs, so every multiply-accumulate is one packed fma.rn.f32x2 (Blackwell's
//     FFMA2: two fp32 FMAs per issue slot) against a broadcast h value;
//   * the four partial sums of a unit meet by a two-stage warp-shuffle reduce-scatter (even lanes end
//     with unit p, odd lanes with unit p + H/2), after which the same threads apply the gates: one
//     block barrier per step;
//   * h lives in shared memory, double-buffered, with each quarter padded by 4 floats so the four
//     lanes of a quad hit distinct banks (conflict-free 128-bit loads);
//   * every global address is a running pointer (no 64-bit multiplies in the loop) and everything a
//     step needs from global memory (input projections, stashed gates, upstream gradients) is
//     prefetched through a shared-memory ring filled with cp.async, in both directions: commit groups complete in
//     order, so cp.async.wait_group pins the prefetch distance.  A register ring of plain loads does not work --
//     the forward's was collapsed to one step by the compiler's scheduler, and the backward's (gru_bwd_kernel, kept
//     for R > 1 rows per CTA and unaligned operands) stalls on memory although it is four visits deep, because every
//     one of its loads shares a scoreboard (see gru_bwd_ring_kernel, the default backward, 69 us against 90 us);
//   * sigmoid / tanh use the ex2 / rcp special-function units (|error| ~ 2e-7, far inside the
//     1e-4 logit tolerance);
//   * inter-layer dropout is NOT applied here: a 30-instruction hash per element inside an in-order
//     step loop costs more than a separate streaming pass (mms_dropout_apply) over the layer output.
// All arithmetic is fp32 (SURVEY §7 hard part 2).
#include "mms_common.cuh"

namespace mms {

constexpr int GRU_MAX_DIRS = 2;
constexpr int PF = 4;   // prefetch distance in time steps

struct GruFwdParams {
    mms_gru_dir_fwd dir[GRU_MAX_DIRS];
    int B;
    float p;
    uint64_t seed, offset;
    const int64_t* offset_dev;
};
struct GruBwdParams {
    mms_gru_dir_bwd dir[GRU_MAX_DIRS];
    int B;
    float p;
    uint64_t seed, offset;
    const int64_t* offset_dev;
};

// sigmoid / tanh on the special-function units: ex2.approx + rcp.approx (2 MUFU ops each).
__device__ __forceinline__ float ex2_ftz(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_ftz(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_sigmoid(float x) { return rcp_ftz(1.f + ex2_ftz(-1.4426950408889634f * x)); }
__device__ __forceinline__ float fast_tanh(float x) { return fmaf(2.f, fast_sigmoid(2.f * x), -1.f); }

__device__ __forceinline__ float ldg_pinned(const float* p) {
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float2 bcast2(float v) { return make_float2(v, v); }

// 16-byte asynchronous global -> shared copy (LDGSTS): the prefetch distance is then fixed by
// cp.async.wait_group and cannot be shortened by the compiler's scheduling of register loads.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// padded position of element k of an H-vector split into quarters of KS floats
template <int KS>
__device__ __forceinline__ int padded(int k) { return k + (k / KS) * 4; }

template <int H, int R>
__global__ void __launch_bounds__(2 * H) gru_fwd_kernel(const GruFwdParams prm) {
    MMS_PDL_TRIGGER();
    constexpr int KS = H / 4, HP = H / 2, HPAD = H + 16;
    const mms_gru_dir_fwd d = prm.dir[blockIdx.y];
    const int tid = threadIdx.x, p = tid >> 2, q = tid & 3;
    const int own = q & 1;                 // which of the two units this lane finishes
    const int ju = p + own * HP;
    const bool first = q < 2;              // first / second lane of the unit (splits the stores)
    const int b0 = blockIdx.x * R;
    const int B = prm.B;
    const int nsteps = d.nsteps;

    __shared__ __align__(16) float hsm[2][R][HPAD];

    // recurrent weights: rows g*H + {p, p+HP}, columns [q*KS, q*KS + KS), packed (unit A, unit B)
    float2 w2[3][KS];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int i = 0; i < KS; ++i)
            w2[g][i] = make_float2(__ldg(d.w_hh + (size_t)(g * H + p) * H + q * KS + i),
                                   __ldg(d.w_hh + (size_t)(g * H + p + HP) * H + q * KS + i));
    float2 bh2[3];
#pragma unroll
    for (int g = 0; g < 3; ++g)
        bh2[g] = q == 0 ? make_float2(__ldg(d.b_hh + g * H + p), __ldg(d.b_hh + g * H + p + HP)) : make_float2(0.f, 0.f);

    for (int i = tid; i < 2 * R * HPAD; i += 2 * H) (&hsm[0][0][0])[i] = 0.f;
    MMS_PDL_WAIT();       // everything above read parameters only; gi / hs / stash belong to the kernels before this one

    const bool do_stash = d.stash != nullptr;

    // running pointers (advance by dt * stride per step); loads clamp the row, stores are guarded
    const int64_t gi_step = (int64_t)d.dt * d.gi_ts, hs_step = (int64_t)d.dt * d.hs_ts, st_step = (int64_t)d.dt * d.st_ts;
    float* hs_p[R];
    float* st_p[R];         // first lane: stash slots 0,1 (r, z); second lane: slots 2,3 (n, W_hn h + b_hn)
    bool live[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int bb = min(b0 + r, B - 1);
        int lv = (b0 + r) < B ? 1 : 0;
        asm volatile("" : "+r"(lv));       // opaque: otherwise the compiler re-derives it from %ctaid and a constant-bank load every step
        live[r] = lv != 0;
        hs_p[r] = d.hs + (int64_t)bb * d.hs_bs + (int64_t)d.t0 * d.hs_ts + ju;
        st_p[r] = do_stash ? d.stash + (int64_t)bb * d.st_bs + (int64_t)d.t0 * d.st_ts + (first ? 0 : 2 * H) + ju : nullptr;
    }
    float* const h_wr = &hsm[0][0][0] + padded<KS>(ju);      // + (buffer * R + r) * HPAD
    uint32_t h_wr_s = (uint32_t)__cvta_generic_to_shared(h_wr);
    asm volatile("" : "+r"(h_wr_s));                        // opaque: keep the address in a register instead of re-deriving it every step

    // Ring of input projections in shared memory, PF steps ahead: threads 0 .. 3H/4-1 each copy 16 bytes
    // of the 3H-float row of step s + PF with cp.async; one commit group per step.
    __shared__ __align__(16) float gsm[PF][R][3 * H];
    constexpr int NCP = 3 * H / 4;
    const float* gi_src[R];
#pragma unroll
    for (int r = 0; r < R; ++r)
        gi_src[r] = d.gi + (int64_t)min(b0 + r, B - 1) * d.gi_bs + (int64_t)d.t0 * d.gi_ts + 4 * (tid < NCP ? tid : 0);
#pragma unroll
    for (int u = 0; u < PF; ++u) {
        if (tid < NCP && u < nsteps) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                cp_async16(&gsm[u][r][4 * tid], gi_src[r]);
                gi_src[r] += gi_step;
            }
        }
        cp_async_commit();
    }
    cp_async_wait<PF - 1>();          // step 0 has landed (for the copying threads); the barrier publishes it
    __syncthreads();

    float hprev[R];
#pragma unroll
    for (int r = 0; r < R; ++r) hprev[r] = 0.f;       // h0 = 0
    static_assert(PF % 2 == 0, "the h double buffer index is the parity of the unrolled step");
    for (int s0 = 0; s0 < nsteps; s0 += PF) {
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            if (s0 + u >= nsteps) break;
            const int cur = u & 1;    // compile-time in the unrolled body (s0 is a multiple of the even PF)
            {   // Refill the slot that was read in the PREVIOUS step (all of its readers are past the barrier that
                // ended that step) with step s - 1 + PF; one commit group per step keeps the group count uniform.
                const int s = s0 + u;
                const int PREV = (u + PF - 1) % PF;
                if (tid < NCP && s >= 1 && s - 1 + PF < nsteps) {
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        cp_async16(&gsm[PREV][r][4 * tid], gi_src[r]);
                        gi_src[r] += gi_step;
                    }
                }
                cp_async_commit();
            }
            float gi[R][3];
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int g = 0; g < 3; ++g) gi[r][g] = gsm[u][r][g * H + ju];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float2 acc[3] = {bh2[0], bh2[1], bh2[2]};
                const float hp = hprev[r];                                     // h_{t-1}[ju]: this thread produced it in the previous step
                const float4* hv = reinterpret_cast<const float4*>(&hsm[cur][r][q * (KS + 4)]);
#pragma unroll
                for (int i4 = 0; i4 < KS / 4; ++i4) {
                    const float4 h4 = hv[i4];
#pragma unroll
                    for (int g = 0; g < 3; ++g) acc[g] = __ffma2_rn(w2[g][4 * i4 + 0], bcast2(h4.x), acc[g]);
#pragma unroll
                    for (int g = 0; g < 3; ++g) acc[g] = __ffma2_rn(w2[g][4 * i4 + 1], bcast2(h4.y), acc[g]);
#pragma unroll
                    for (int g = 0; g < 3; ++g) acc[g] = __ffma2_rn(w2[g][4 * i4 + 2], bcast2(h4.z), acc[g]);
#pragma unroll
                    for (int g = 0; g < 3; ++g) acc[g] = __ffma2_rn(w2[g][4 * i4 + 3], bcast2(h4.w), acc[g]);
                }
                // reduce-scatter over the quad: stage 1 keeps this lane's unit, stage 2 completes it
                float sg[3];
#pragma unroll
                for (int g = 0; g < 3; ++g) {
                    const float keep = own ? acc[g].y : acc[g].x;
                    const float send = own ? acc[g].x : acc[g].y;
                    sg[g] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
                }
#pragma unroll
                for (int g = 0; g < 3; ++g) sg[g] += __shfl_xor_sync(0xffffffffu, sg[g], 2);
                // sg = W_h{r,z,n} h + b_h{r,z,n} of unit ju
                const float rg = fast_sigmoid(sg[0] + gi[r][0]);
                const float zg = fast_sigmoid(sg[1] + gi[r][1]);
                const float ng = fast_tanh(fmaf(rg, sg[2], gi[r][2]));
                const float hn = fmaf(zg, hp - ng, ng);                        // (1-z)*n + z*h
                hprev[r] = hn;
                if (first)                                                     // predicated store, no branch; the next step waits on it
                    asm volatile("st.shared.f32 [%0], %1;" ::"r"(h_wr_s + (uint32_t)(((cur ^ 1) * R + r) * HPAD * 4)), "f"(hn) : "memory");
                if (first && live[r]) *hs_p[r] = hn;
                if (do_stash && live[r]) {                                     // uniform, predicated stores
                    st_p[r][0] = first ? rg : ng;
                    st_p[r][H] = first ? zg : sg[2];
                }
                hs_p[r] += hs_step;
                st_p[r] += st_step;
            }
            cp_async_wait<PF - 2>();      // the copies for step s + 1 are complete for the copying threads ...
            __syncthreads();              // ... and, with h[cur^1], visible to every thread
        }
    }
}

template <int H, int R>
__global__ void __launch_bounds__(2 * H) gru_bwd_kernel(const GruBwdParams prm) {
    constexpr int KS = H / 4, HP = H / 2, GP = H + 16;      // GP: padded length of one gate vector
    constexpr int PFB = R == 1 ? 4 : 2;                     // shallower prefetch ring when several rows share the registers
    const mms_gru_dir_bwd d = prm.dir[blockIdx.y];
    const int tid = threadIdx.x, p = tid >> 2, q = tid & 3;
    const int own = q & 1;
    const int ku = p + own * HP;           // the column (hidden unit) whose gate math this lane does
    const bool first = q < 2;
    const int b0 = blockIdx.x * R;
    const int B = prm.B;
    const int nsteps = d.nsteps;

    __shared__ __align__(16) float dgh[2][R][3 * GP];

    // columns {p, p+HP} of W_hh, gate rows [g*H + q*KS, +KS), packed (column A, column B)
    float2 w2[3][KS];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int i = 0; i < KS; ++i)
            w2[g][i] = make_float2(__ldg(d.w_hh + (size_t)(g * H + q * KS + i) * H + p),
                                   __ldg(d.w_hh + (size_t)(g * H + q * KS + i) * H + p + HP));

    const bool has_dout = d.dout != nullptr;

    // The visit order is the reverse of the forward order: forward step s = nsteps-1 ... 0 at time
    // t = t0 + s*dt.  Running pointers start at the last forward step and move by -dt * stride.
    const int t_last = d.t0 + (nsteps - 1) * d.dt;
    const int64_t st_step = -(int64_t)d.dt * d.st_ts, hs_step = -(int64_t)d.dt * d.hs_ts;
    const int64_t do_step = -(int64_t)d.dt * d.do_ts, d_step = -(int64_t)d.dt * d.d_ts;
    const float* st_p[R];     // prefetch side (PF visits ahead)
    const float* hp_p[R];     // h_{prev} of the prefetched step
    const float* do_p[R];
    float* D_p[R];            // store side (current visit)
    float dh[R];
    float dlast[R];
    bool live[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int bb = min(b0 + r, B - 1);
        live[r] = (b0 + r) < B;
        st_p[r] = d.stash + (int64_t)bb * d.st_bs + (int64_t)t_last * d.st_ts + ku;
        hp_p[r] = d.hs + (int64_t)bb * d.hs_bs + (int64_t)(t_last - d.dt) * d.hs_ts + ku;   // only read when s > 0
        do_p[r] = has_dout ? d.dout + (int64_t)bb * d.do_bs + (int64_t)t_last * d.do_ts + ku : nullptr;
        D_p[r] = d.D + (int64_t)bb * d.d_bs + (int64_t)t_last * d.d_ts + (first ? 0 : 2 * H) + ku;
        dlast[r] = d.dout_last ? __ldg(d.dout_last + (int64_t)bb * d.dl_ld + ku) : 0.f;
        // initial recurrent gradient: optional projection of the head gradient (dlast = dhid @ W0)
        float s = 0.f;
        if (d.dh_head) {
            for (int i = 0; i < HEAD_HID; ++i)
                s = fmaf(__ldg(d.dh_head + (size_t)bb * HEAD_HID + i), __ldg(d.w0 + (size_t)i * d.w0_ld + d.w0_col + ku), s);
        }
        dh[r] = s;
    }

    float* const g_wr = &dgh[0][0][0] + padded<KS>(ku);     // + (buffer * R + r) * 3 * GP

    // ring of per-step inputs for column ku: stash (r,z,n,qq), h_prev, dout
    struct StepIn { float r, z, n, qq, hp, dout; };
    StepIn ring[PFB][R];
    int fetch_s = nsteps - 1;         // forward-step index the prefetch pointers refer to
    auto fetch = [&](int r) {
        StepIn v;
        const float* sp = st_p[r];
        // volatile asm: the loads are issued HERE, PFB visits ahead of their use; a plain __ldg is sunk towards its use by
        // ptxas whenever it decides to save registers, which collapses the ring and exposes the global-load latency
        v.r = ldg_pinned(sp);
        v.z = ldg_pinned(sp + H);
        v.n = ldg_pinned(sp + 2 * H);
        v.qq = ldg_pinned(sp + 3 * H);
        v.hp = fetch_s > 0 ? ldg_pinned(hp_p[r]) : 0.f;
        v.dout = has_dout ? ldg_pinned(do_p[r]) : 0.f;
        return v;
    };
    auto advance = [&]() {            // move the prefetch pointers one visit further (if any step is left)
        if (fetch_s > 0) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                st_p[r] += st_step;
                hp_p[r] += hs_step;
                if (has_dout) do_p[r] += do_step;
            }
        }
        --fetch_s;
    };
#pragma unroll
    for (int u = 0; u < PFB; ++u) {
#pragma unroll
        for (int r = 0; r < R; ++r) ring[u][r] = fetch_s >= 0 ? fetch(r) : StepIn{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        advance();
    }

    const int v_extra = d.dl_at_first ? nsteps - 1 : 0;     // visit at which dout_last is added
    int buf = 0;      // kept a run-time value on purpose: with a compile-time parity ptxas settles on 168 registers and a
                      // schedule that measured 127 us per launch instead of 90 us
    for (int v0 = 0; v0 < nsteps; v0 += PFB) {
#pragma unroll
        for (int u = 0; u < PFB; ++u) {
            const int v = v0 + u;
            if (v >= nsteps) break;
            const int s = nsteps - 1 - v;
            StepIn in[R];
#pragma unroll
            for (int r = 0; r < R; ++r) in[r] = ring[u][r];
            if (fetch_s >= 0) {
#pragma unroll
                for (int r = 0; r < R; ++r) ring[u][r] = fetch(r);
            }
            advance();
            float dhz[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const StepIn& x = in[r];
                const float dht = dh[r] + x.dout + (v == v_extra ? dlast[r] : 0.f);
                const float dn = dht * (1.f - x.z);
                const float dz = dht * (x.hp - x.n);
                const float dnp = dn * (1.f - x.n * x.n);
                const float dq = dnp * x.r;
                const float dr = dnp * x.qq;
                const float dzp = dz * x.z * (1.f - x.z);
                const float drp = dr * x.r * (1.f - x.r);
                dhz[r] = dht * x.z;
                if (first) {
                    float* g = g_wr + (buf * R + r) * 3 * GP;
                    g[0] = drp; g[GP] = dzp; g[2 * GP] = dq;
                }
                if (live[r]) {          // D = (d r_pre, d z_pre, d n_pre, d q): first lane stores 0,1; second 2,3
                    D_p[r][0] = first ? drp : dnp;
                    D_p[r][H] = first ? dzp : dq;
                }
                D_p[r] += d_step;
            }
            __syncthreads();
            if (s > 0) {     // the gradient flowing into h_{-1} = h0 is not needed
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    float2 acc[3] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
                    for (int g = 0; g < 3; ++g) {
                        const float4* gv = reinterpret_cast<const float4*>(&dgh[buf][r][g * GP + q * (KS + 4)]);
#pragma unroll
                        for (int i4 = 0; i4 < KS / 4; ++i4) {
                            const float4 g4 = gv[i4];
                            acc[g] = __ffma2_rn(w2[g][4 * i4 + 0], bcast2(g4.x), acc[g]);
                            acc[g] = __ffma2_rn(w2[g][4 * i4 + 1], bcast2(g4.y), acc[g]);
                            acc[g] = __ffma2_rn(w2[g][4 * i4 + 2], bcast2(g4.z), acc[g]);
                            acc[g] = __ffma2_rn(w2[g][4 * i4 + 3], bcast2(g4.w), acc[g]);
                        }
                    }
                    const float ax = (acc[0].x + acc[1].x) + acc[2].x, ay = (acc[0].y + acc[1].y) + acc[2].y;
                    float t = (own ? ay : ax) + __shfl_xor_sync(0xffffffffu, own ? ax : ay, 1);
                    t += __shfl_xor_sync(0xffffffffu, t, 2);
                    dh[r] = dhz[r] + t;
                }
            }
            buf ^= 1;
        }
    }
}

// Backward recurrence with the per-visit inputs staged through a shared-memory ring (one batch row per CTA).
//
// Why a second variant: in gru_bwd_kernel the six values a visit needs travel through a register ring of plain global
// loads.  ptxas gives every one of those LDGs the SAME scoreboard (decoded from the SASS control words: all 24 ring loads
// write SB5), and a scoreboard wait is a wait for its counter to reach zero, i.e. for the YOUNGEST load in flight -- so the
// consumer of the 4-visits-old slot also waits for the slot that was refilled a moment ago (in one of the four unrolled
// visits literally: a register move the allocator inserted after the refill), and the nominal prefetch distance of four
// visits collapses to one or less (ncu: 35-39 % of the stall samples are long_scoreboard, on two instructions of the four
// unrolled visits).  cp.async (LDGSTS) completion is tracked by commit groups instead of scoreboards, groups complete in
// order and cp.async.wait_group N only waits for the groups older than the N youngest: a true ring.  Threads 0 .. 6H/4-1
// copy 16 bytes each of the visit's row (stash 4H | h_prev H | dout H) PF-1 visits ahead; the barrier every visit already
// has publishes the slot, and the six scalars of visit v+1 are read from shared memory into registers right after the
// barrier of visit v, behind the mat-vec, so no shared-memory round trip is added to the dependent chain.
//
// Everything that is invariant over the visits (roles, shared-memory addresses, strides, step counts) is computed once
// and made opaque to the compiler: at ~170 registers ptxas otherwise re-derives such values inside every visit from
// %tid / %ctaid / constant-bank loads (S2R, LDC and S2UR + LEA chains between the barrier and the loads of the mat-vec),
// which is what made the earlier register-lean variants slower than the 254-register kernel.  Shared memory is
// addressed through 32-bit window addresses with immediate offsets, stores to the gate buffer are unconditional (the
// two lanes that finish the same unit store the same value), copies are predicated instead of branched around.
__device__ __forceinline__ float lds_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float4 lds_v4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
// predicated 16-byte asynchronous copy: no branch around the LDGSTS
__device__ __forceinline__ void cp_async16_if(uint32_t smem_dst, const void* gmem_src, int pred) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p cp.async.cg.shared.global [%0], [%1], 16;\n\t}" ::"r"(smem_dst), "l"(gmem_src),
                 "r"(pred)
                 : "memory");
}
#define MMS_OPAQUE32(x) asm volatile("" : "+r"(x))
#define MMS_OPAQUE64(x) asm volatile("" : "+l"(x))
#define MMS_OPAQUEF(x) asm volatile("" : "+f"(x))

template <int H, int PF>
__global__ void __launch_bounds__(2 * H) gru_bwd_ring_kernel(const GruBwdParams prm) {
    MMS_PDL_TRIGGER();
    constexpr int KS = H / 4, HP = H / 2, GP = H + 16;      // GP: padded length of one gate vector
    constexpr int ROW = 6 * H;                              // floats per ring slot: r, z, n, q | h_prev | dout
    constexpr int NCP = ROW / 4;                            // 16-byte chunks per slot, one per copying thread
    static_assert(PF % 2 == 0 && PF >= 4, "the gate double-buffer index is the parity of the unrolled visit");
    static_assert(NCP <= 2 * H, "one chunk per thread");
    const mms_gru_dir_bwd d = prm.dir[blockIdx.y];
    const int tid = threadIdx.x, p = tid >> 2, q = tid & 3;
    const int own = q & 1;
    const int ku = p + own * HP;           // the column (hidden unit) whose gate math this lane does
    const bool first = q < 2;
    const int bb = blockIdx.x;             // one batch row per CTA: grid.x == B
    int nsteps = d.nsteps;
    MMS_OPAQUE32(nsteps);

    __shared__ __align__(16) float dgh[2][3 * GP];
    __shared__ __align__(16) float ring[PF][ROW];

    // columns {p, p+HP} of W_hh, gate rows [g*H + q*KS, +KS), packed (column A, column B)
    float2 w2[3][KS];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int i = 0; i < KS; ++i)
            w2[g][i] = make_float2(__ldg(d.w_hh + (size_t)(g * H + q * KS + i) * H + p),
                                   __ldg(d.w_hh + (size_t)(g * H + q * KS + i) * H + p + HP));

    MMS_PDL_WAIT();       // the weights above are parameters; stash / hs / dout / dh_head belong to the kernels before this one
    int has_dout = d.dout != nullptr ? 1 : 0;
    MMS_OPAQUE32(has_dout);
    // visit v handles forward step s = nsteps-1-v at time t_last - v*dt
    const int t_last = d.t0 + (nsteps - 1) * d.dt;

    // copy role of this thread: chunk tid of the row.  Threads without a role keep a valid pointer that is never read.
    int copier = 0, is_hp = 0;
    const float* src = d.stash;
    int64_t sstep = 0;
    if (tid < H) {
        copier = 1; src = d.stash + (int64_t)bb * d.st_bs + (int64_t)t_last * d.st_ts + 4 * tid; sstep = -(int64_t)d.dt * d.st_ts;
    } else if (tid < H + H / 4) {
        copier = 1; is_hp = 1;
        src = d.hs + (int64_t)bb * d.hs_bs + (int64_t)(t_last - d.dt) * d.hs_ts + 4 * (tid - H); sstep = -(int64_t)d.dt * d.hs_ts;
    } else if (tid < NCP && has_dout) {
        copier = 1; src = d.dout + (int64_t)bb * d.do_bs + (int64_t)t_last * d.do_ts + 4 * (tid - H - H / 4); sstep = -(int64_t)d.dt * d.do_ts;
    }
    // h_prev of the first forward step (= the last visit) is h0 = 0, not memory: copies of h_prev stop one visit early
    int n_copy = is_hp ? nsteps - 1 : nsteps;
    if (!copier) n_copy = 0;
    MMS_OPAQUE32(n_copy);
    MMS_OPAQUE64(sstep);
    uint32_t ring_wr_s = (uint32_t)__cvta_generic_to_shared(&ring[0][0]) + 16u * (uint32_t)tid;
    uint32_t ring_rd_s = (uint32_t)__cvta_generic_to_shared(&ring[0][0]) + 4u * (uint32_t)ku;
    uint32_t g_wr_s = (uint32_t)__cvta_generic_to_shared(&dgh[0][0]) + 4u * (uint32_t)padded<KS>(ku);
    uint32_t g_rd_s = (uint32_t)__cvta_generic_to_shared(&dgh[0][0]) + 4u * (uint32_t)(q * (KS + 4));
    MMS_OPAQUE32(ring_wr_s);
    MMS_OPAQUE32(ring_rd_s);
    MMS_OPAQUE32(g_wr_s);
    MMS_OPAQUE32(g_rd_s);

    // the copies of visit w go to slot w % PF (compile-time at every call site)
#define MMS_RING_ISSUE(w, slot)                                                       \
    do {                                                                              \
        cp_async16_if(ring_wr_s + (uint32_t)((slot) * ROW * 4), src, (w) < n_copy);   \
        src += sstep;                                                                 \
    } while (0)

#pragma unroll
    for (int u = 0; u < PF; ++u) {
        MMS_RING_ISSUE(u, u);
        cp_async_commit();
    }

    float* D_p = d.D + (int64_t)bb * d.d_bs + (int64_t)t_last * d.d_ts + (first ? 0 : 2 * H) + ku;
    int64_t d_step = -(int64_t)d.dt * d.d_ts;
    MMS_OPAQUE64(d_step);
    float dlast = d.dout_last ? __ldg(d.dout_last + (int64_t)bb * d.dl_ld + ku) : 0.f;
    // initial recurrent gradient: optional projection of the head gradient (dhid @ W0)
    float dh = 0.f;
    if (d.dh_head) {
        for (int i = 0; i < HEAD_HID; ++i)
            dh = fmaf(__ldg(d.dh_head + (size_t)bb * HEAD_HID + i), __ldg(d.w0 + (size_t)i * d.w0_ld + d.w0_col + ku), dh);
    }
    int v_extra = d.dl_at_first ? nsteps - 1 : 0;           // visit at which dout_last is added
    MMS_OPAQUE32(v_extra);
    MMS_OPAQUEF(dlast);
    int sel_first = first ? 1 : 0, sel_own = own;
    MMS_OPAQUE32(sel_first);
    MMS_OPAQUE32(sel_own);

    // What the dependent chain of a visit needs is dht = dh + (dout [+ dout_last]) and then one multiply per output:
    //   d r_pre = dht * cr,  d z_pre = dht * cz,  d n_pre = dht * cn,  d q = dht * cq,  dh_next = dht * z + W^T (...)
    // with coefficients that depend only on the stashed gates.  They are formed from the ring slot of visit v+1 behind the
    // mat-vec of visit v (off the chain), which leaves FADD -> FMUL -> STS between the last shuffle and the barrier.
    struct StepIn { float add, cr, cz, cn, cq, z; };
#define MMS_RING_LOAD(dst, slot, vn)                                                  \
    do {                                                                              \
        const uint32_t a_ = ring_rd_s + (uint32_t)((slot) * ROW * 4);                 \
        const float r_ = lds_f32(a_), z_ = lds_f32(a_ + 4 * H), n_ = lds_f32(a_ + 8 * H), q_ = lds_f32(a_ + 12 * H); \
        const float hpl_ = lds_f32(a_ + 16 * H), dol_ = lds_f32(a_ + 20 * H);         \
        const float hp_ = (vn) < nsteps - 1 ? hpl_ : 0.f;      /* h_prev of forward step 0 is h0 = 0 */ \
        const float cn_ = (1.f - z_) * (1.f - n_ * n_);                               \
        dst.add = (has_dout ? dol_ : 0.f) + ((vn) == v_extra ? dlast : 0.f);          \
        dst.cn = cn_;                                                                 \
        dst.cq = cn_ * r_;                                                            \
        dst.cr = cn_ * q_ * (r_ * (1.f - r_));                                        \
        dst.cz = (hp_ - n_) * (z_ * (1.f - z_));                                      \
        dst.z = z_;                                                                   \
    } while (0)

    cp_async_wait<PF - 1>();          // visit 0 has landed (for the copying threads); the barrier publishes it
    __syncthreads();
    StepIn nx;
    MMS_RING_LOAD(nx, 0, 0);

    for (int v0 = 0; v0 < nsteps; v0 += PF) {
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            const int v = v0 + u;
            if (v >= nsteps) break;
            const int cur = u & 1;    // compile-time in the unrolled body (v0 is a multiple of the even PF)
            const StepIn x = nx;
            const float dht = dh + x.add;
            const float drp = dht * x.cr, dzp = dht * x.cz, dnp = dht * x.cn, dq = dht * x.cq;
            const float dhz = dht * x.z;
            {   // both lanes that finish unit ku hold the same three values: unconditional stores, no branch
                const uint32_t g = g_wr_s + (uint32_t)(cur * 3 * GP * 4);
                sts_f32(g, drp);
                sts_f32(g + GP * 4, dzp);
                sts_f32(g + 2 * GP * 4, dq);
            }
            // D = (d r_pre, d z_pre, d n_pre, d q): first lane stores 0,1; second 2,3
            D_p[0] = sel_first ? drp : dnp;
            D_p[H] = sel_first ? dzp : dq;
            D_p += d_step;
            cp_async_wait<PF - 2>();      // the copies for visit v + 1 are complete for the copying threads ...
            __syncthreads();              // ... and, with the gate buffer `cur`, visible to every thread
            if (v + 1 < nsteps) {         // the gradient flowing into h_{-1} = h0 is not needed
                // Slot u held THIS visit's inputs; every thread read them before it arrived at the barrier above, so the
                // slot is free: refill it with visit v + PF.  One commit group per visit keeps the group count uniform.
                MMS_RING_ISSUE(v + PF, u);
                cp_async_commit();
                float2 acc[3] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
                for (int g = 0; g < 3; ++g) {
                    const uint32_t ga = g_rd_s + (uint32_t)((cur * 3 * GP + g * GP) * 4);
#pragma unroll
                    for (int i4 = 0; i4 < KS / 4; ++i4) {
                        const float4 g4 = lds_v4(ga + 16 * i4);
                        acc[g] = __ffma2_rn(w2[g][4 * i4 + 0], bcast2(g4.x), acc[g]);
                        acc[g] = __ffma2_rn(w2[g][4 * i4 + 1], bcast2(g4.y), acc[g]);
                        acc[g] = __ffma2_rn(w2[g][4 * i4 + 2], bcast2(g4.z), acc[g]);
                        acc[g] = __ffma2_rn(w2[g][4 * i4 + 3], bcast2(g4.w), acc[g]);
                    }
                }
                MMS_RING_LOAD(nx, (u + 1) % PF, v + 1);      // next visit's inputs, behind the mat-vec
                const float ax = (acc[0].x + acc[1].x) + acc[2].x, ay = (acc[0].y + acc[1].y) + acc[2].y;
                float t = (sel_own ? ay : ax) + __shfl_xor_sync(0xffffffffu, sel_own ? ax : ay, 1);
                t += __shfl_xor_sync(0xffffffffu, t, 2);
                dh = dhz + t;
            }
        }
    }
#undef MMS_RING_ISSUE
#undef MMS_RING_LOAD
}

// Forward recurrence, second version (the default since round 2: 68 -> 57 us per launch on a B200; MMS_GRU_FWD_V2=0 restores the
// first; one batch row per CTA).  Same algorithm and data movement as gru_fwd_kernel, three changes aimed at the dependent chain of a
// step (ncu: 36 % fixed-latency waits, 21 % short scoreboard, 4 % branch resolving on one warp per scheduler):
//   * thread (j, q) = (tid >> 1, tid & 1) owns ONE hidden unit and half of the reduction index, so the partial sums meet in
//     ONE shuffle stage instead of two.  FFMA2 packing: (r, z) gate weights of the unit against a broadcast h_k, and the n
//     gate over pairs of k against (h_k, h_k+1); the (r, z) chain is split in two accumulators to keep three 16-deep chains;
//   * -log2(e) is folded into W_h{r,z}, b_h{r,z} and (off the chain) into the input projections, -2 log2(e) into the n gate:
//     sigma(x) = 1 / (1 + 2^x') and tanh(a) = 2 / (1 + 2^a'') - 1 lose the multiplies in front of ex2;
//   * both lanes of a unit hold the same h: the shared-memory store is unconditional, global stores are predicated by
//     selects -- no divergent branch in the loop; every loop invariant is pinned (see gru_bwd_ring_kernel).
// The stashed W_hn h + b_hn is un-scaled again off the chain (one rounding, ~1e-7 relative).
template <int H>
__global__ void __launch_bounds__(2 * H) gru_fwd_v2_kernel(const GruFwdParams prm) {
    MMS_PDL_TRIGGER();
    constexpr int KH = H / 2;                 // reduction elements per thread
    constexpr int HPAD = H + 8;               // two halves, each padded by 4 floats (distinct banks for the two lanes of a unit)
    constexpr float C1 = -1.4426950408889634f, C2 = 2.f * C1, INV_C2 = 1.f / C2;
    static_assert(KH % 4 == 0, "float4 reads of h");
    const mms_gru_dir_fwd d = prm.dir[blockIdx.y];
    const int tid = threadIdx.x, j = tid >> 1, q = tid & 1;
    const int bb = blockIdx.x;                // one batch row per CTA: grid.x == B
    int nsteps = d.nsteps;
    MMS_OPAQUE32(nsteps);

    __shared__ __align__(16) float hsm[2][HPAD];
    __shared__ __align__(16) float gsm[PF][3 * H];

    // recurrent weights of unit j, columns [q*KH, q*KH + KH), pre-scaled
    float2 w_rz[KH];      // (W_hr, W_hz)[j][k] * C1
    float2 w_n[KH / 2];   // (W_hn[j][2i], W_hn[j][2i+1]) * C2
#pragma unroll
    for (int i = 0; i < KH; ++i)
        w_rz[i] = make_float2(C1 * __ldg(d.w_hh + (size_t)(0 * H + j) * H + q * KH + i), C1 * __ldg(d.w_hh + (size_t)(1 * H + j) * H + q * KH + i));
#pragma unroll
    for (int i = 0; i < KH / 2; ++i)
        w_n[i] = make_float2(C2 * __ldg(d.w_hh + (size_t)(2 * H + j) * H + q * KH + 2 * i),
                             C2 * __ldg(d.w_hh + (size_t)(2 * H + j) * H + q * KH + 2 * i + 1));
    const float2 b_rz = q == 0 ? make_float2(C1 * __ldg(d.b_hh + j), C1 * __ldg(d.b_hh + H + j)) : make_float2(0.f, 0.f);
    const float2 b_n = q == 0 ? make_float2(C2 * __ldg(d.b_hh + 2 * H + j), 0.f) : make_float2(0.f, 0.f);

    for (int i = tid; i < 2 * HPAD; i += 2 * H) (&hsm[0][0])[i] = 0.f;        // h0 = 0
    MMS_PDL_WAIT();       // parameters only above

    int do_stash = d.stash != nullptr ? 1 : 0;
    MMS_OPAQUE32(do_stash);
    int64_t hs_step = (int64_t)d.dt * d.hs_ts, st_step = (int64_t)d.dt * d.st_ts, gi_step = (int64_t)d.dt * d.gi_ts;
    MMS_OPAQUE64(hs_step);
    MMS_OPAQUE64(st_step);
    MMS_OPAQUE64(gi_step);
    float* hs_p = d.hs + (int64_t)bb * d.hs_bs + (int64_t)d.t0 * d.hs_ts + j;
    // lane 0 of a unit stores stash slots 0, 1 (r, z); lane 1 stores slots 2, 3 (n, W_hn h + b_hn).  Without a stash the
    // pointer stays valid (the h row) and is never written.
    float* st_p = do_stash ? d.stash + (int64_t)bb * d.st_bs + (int64_t)d.t0 * d.st_ts + (q ? 2 * H : 0) + j : hs_p;
    int q0 = q == 0 ? 1 : 0;
    MMS_OPAQUE32(q0);

    uint32_t h_wr_s = (uint32_t)__cvta_generic_to_shared(&hsm[0][0]) + 4u * (uint32_t)(j + (j / KH) * 4);
    uint32_t h_rd_s = (uint32_t)__cvta_generic_to_shared(&hsm[0][0]) + 4u * (uint32_t)(q * (KH + 4));
    uint32_t g_rd_s = (uint32_t)__cvta_generic_to_shared(&gsm[0][0]) + 4u * (uint32_t)j;
    uint32_t g_wr_s = (uint32_t)__cvta_generic_to_shared(&gsm[0][0]) + 16u * (uint32_t)tid;
    MMS_OPAQUE32(h_wr_s);
    MMS_OPAQUE32(h_rd_s);
    MMS_OPAQUE32(g_rd_s);
    MMS_OPAQUE32(g_wr_s);

    // ring of input projections: threads 0 .. 3H/4-1 copy 16 bytes each of the 3H-float row of a step, PF steps ahead
    constexpr int NCP = 3 * H / 4;
    const float* gi_src = d.gi + (int64_t)bb * d.gi_bs + (int64_t)d.t0 * d.gi_ts + 4 * (tid < NCP ? tid : 0);
    int n_copy = tid < NCP ? nsteps : 0;
    MMS_OPAQUE32(n_copy);
#pragma unroll
    for (int u = 0; u < PF; ++u) {
        cp_async16_if(g_wr_s + (uint32_t)(u * 3 * H * 4), gi_src, u < n_copy);
        gi_src += gi_step;
        cp_async_commit();
    }
    cp_async_wait<PF - 1>();          // step 0 has landed (for the copying threads); the barrier publishes it (and h0)
    __syncthreads();

    float hprev = 0.f;
    float p_h = 0.f, p_a = 0.f, p_b = 0.f;        // h and the two stash values of the previous step, stored one step late
    static_assert(PF % 2 == 0, "the h double buffer index is the parity of the unrolled step");
    for (int s0 = 0; s0 < nsteps; s0 += PF) {
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            const int s = s0 + u;
            if (s >= nsteps) break;
            const int cur = u & 1;    // compile-time in the unrolled body
            // pre-scaled input projections of this step (available long before the reduction ends)
            const uint32_t ga = g_rd_s + (uint32_t)(u * 3 * H * 4);
            const float g_r = C1 * lds_f32(ga), g_z = C1 * lds_f32(ga + 4 * H), g_n = C2 * lds_f32(ga + 8 * H);
            float2 a0 = b_rz, a1 = make_float2(0.f, 0.f), an = b_n;
            const uint32_t ha = h_rd_s + (uint32_t)(cur * HPAD * 4);
#pragma unroll
            for (int i4 = 0; i4 < KH / 4; ++i4) {
                const float4 h4 = lds_v4(ha + 16 * i4);
                a0 = __ffma2_rn(w_rz[4 * i4 + 0], bcast2(h4.x), a0);
                a1 = __ffma2_rn(w_rz[4 * i4 + 1], bcast2(h4.y), a1);
                an = __ffma2_rn(w_n[2 * i4 + 0], make_float2(h4.x, h4.y), an);
                a0 = __ffma2_rn(w_rz[4 * i4 + 2], bcast2(h4.z), a0);
                a1 = __ffma2_rn(w_rz[4 * i4 + 3], bcast2(h4.w), a1);
                an = __ffma2_rn(w_n[2 * i4 + 1], make_float2(h4.z, h4.w), an);
            }
            // The global stores of the PREVIOUS step go out here, behind the shared-memory loads of the mat-vec: nothing in
            // the recurrence depends on them, so they must not sit between a barrier and the loads that follow it.
            if (s > 0) {
                if (q0) *hs_p = p_h;
                if (do_stash) {
                    st_p[0] = p_a;
                    st_p[H] = p_b;
                }
                hs_p += hs_step;
                st_p += st_step;
            }
            float sr = a0.x + a1.x, sz = a0.y + a1.y, sn = an.x + an.y;
            sr += __shfl_xor_sync(0xffffffffu, sr, 1);
            sz += __shfl_xor_sync(0xffffffffu, sz, 1);
            sn += __shfl_xor_sync(0xffffffffu, sn, 1);
            // sr, sz = C1 * (W_h{r,z} h + b_h{r,z}); sn = C2 * (W_hn h + b_hn)
            const float rg = rcp_ftz(1.f + ex2_ftz(sr + g_r));
            const float zg = rcp_ftz(1.f + ex2_ftz(sz + g_z));
            const float sg = rcp_ftz(1.f + ex2_ftz(fmaf(rg, sn, g_n)));
            const float ng = fmaf(2.f, sg, -1.f);
            const float hn = fmaf(zg, hprev - ng, ng);                        // (1-z)*n + z*h
            hprev = hn;
            sts_f32(h_wr_s + (uint32_t)((cur ^ 1) * HPAD * 4), hn);           // both lanes of the unit: same value, same address
            cp_async_wait<PF - 2>();      // the copies for step s + 1 are complete for the copying threads ...
            __syncthreads();              // ... and, with h[cur^1], visible to every thread
            p_h = hn;
            p_a = q0 ? rg : ng;
            p_b = q0 ? zg : sn * INV_C2;
            // every thread has read slot u (before the barrier): refill it with step s + PF; one commit group per step
            cp_async16_if(g_wr_s + (uint32_t)(u * 3 * H * 4), gi_src, s + PF < n_copy);
            gi_src += gi_step;
            cp_async_commit();
        }
    }
    // the last step's outputs (nsteps >= 1)
    if (q0) *hs_p = p_h;
    if (do_stash) {
        st_p[0] = p_a;
        st_p[H] = p_b;
    }
}

static inline int rows_per_cta(int B, int ndirs) {
    // one row per CTA while all CTAs fit in ~2 waves on 148 SMs; more rows per CTA beyond that
    int R = 1;
    while (R < 4 && (int64_t)cdiv(B, R) * ndirs > 296) R *= 2;
    return R;
}

// Hidden size 128 runs the same kernels as 32 / 64, instantiated at H = 128 (256 threads, one CTA per SM):
//   gru_fwd_v2_kernel<128>        ptxas: 244 registers, no spill; static shared memory 4 x 3H (ring) + 2 x (H + 8) floats = 7232 bytes
//   gru_bwd_ring_kernel<128, 8>   ptxas: 255 registers, no spill; 8 x 6H (ring) + 2 x 3 x (H + 16) floats = 28032 bytes
//   gru_bwd_ring_kernel<128, 4>   ptxas: 255 registers, no spill; 4 x 6H + 2 x 3 x (H + 16) floats = 15744 bytes
// 256 threads x 255 registers = 65280 of the SM's 65536: one recurrence CTA per SM.  W_hh of one direction (3H x H fp32 =
// 192 KB) lives entirely in registers, 192 floats per thread.  The multi-row kernels (gru_fwd_kernel / gru_bwd_kernel with
// R > 1) spill at H = 128 (gru_bwd_kernel<128, 1> already spills 96 bytes), so they are not instantiated: large batches run one
// row per CTA over several waves, and the register-ring backward (GRU_BWD_RING=0, or operands that are not 16-byte aligned) is
// refused at this size.
constexpr int GRU_H_WIDE = 128;

template <int H>
static int gru_fwd_dispatch(const GruFwdParams& prm, int ndirs, cudaStream_t st) {
    const bool wide = H == GRU_H_WIDE;
    const int R = wide ? 1 : rows_per_cta(prm.B, ndirs);          // hidden size 128: one row per CTA at every batch size
    dim3 grid(cdiv(prm.B, R), ndirs);
    MMS_REQUIRE(!wide || option_get("GRU_FWD_V2", 1) == 1,
                "gru_recur_fwd: GRU_FWD_V2=0 selects the multi-row forward, which has no hidden size %d kernel", H);
    if (R == 1 && option_get("GRU_FWD_V2", 1) == 1) {      // experiment (see gru_fwd_v2_kernel)
        MMS_PROF_BEGIN(st);
        auto k2 = gru_fwd_v2_kernel<H>;
        MMS_LAUNCH(k2, grid, dim3(2 * H), 0, st, prm);
        MMS_LAUNCH_CHECK("gru_fwd_v2_kernel");
        return MMS_OK;
    }
    if constexpr (H != GRU_H_WIDE) {
        MMS_PROF_BEGIN(st);
        auto k1 = gru_fwd_kernel<H, 1>;
        auto k2 = gru_fwd_kernel<H, 2>;
        auto k4 = gru_fwd_kernel<H, 4>;
        if (R == 1) MMS_LAUNCH(k1, grid, dim3(2 * H), 0, st, prm);
        else if (R == 2) MMS_LAUNCH(k2, grid, dim3(2 * H), 0, st, prm);
        else MMS_LAUNCH(k4, grid, dim3(2 * H), 0, st, prm);
        MMS_LAUNCH_CHECK("gru_fwd_kernel");
    }
    return MMS_OK;
}

// the shared-memory-ring variant copies whole 16-byte pieces of the stash / h / dout rows
static bool bwd_ring_ok(const GruBwdParams& prm, int ndirs) {
    auto ok = [](const void* p, int64_t bs, int64_t ts) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && bs % 4 == 0 && ts % 4 == 0; };
    for (int i = 0; i < ndirs; ++i) {
        const mms_gru_dir_bwd& d = prm.dir[i];
        if (!ok(d.stash, d.st_bs, d.st_ts) || !ok(d.hs, d.hs_bs, d.hs_ts)) return false;
        if (d.dout && !ok(d.dout, d.do_bs, d.do_ts)) return false;
    }
    return true;
}

template <int H>
static int gru_bwd_dispatch(const GruBwdParams& prm, int ndirs, cudaStream_t st) {
    const int R = H == GRU_H_WIDE ? 1 : rows_per_cta(prm.B, ndirs);   // hidden size 128: one row per CTA at every batch size
    dim3 grid(cdiv(prm.B, R), ndirs);
    // MMS_GRU_BWD_RING / mms_set_option("GRU_BWD_RING", n): shared-memory ring of depth 8 (default) or 4; 0 = the register-ring
    // kernel (gru_bwd_kernel), which also serves R > 1 rows per CTA and operands that are not 16-byte aligned.
    // Measured on a B200 (profiles/r1_ab_gru_bwd_ring.json): 89.6 us (register ring) -> 69.3 us (depth 4) -> 66.7 us (depth 8)
    // per launch; depth 8 is the default since round 2 (the whole GPU suite runs with it).
    const int ring = option_get("GRU_BWD_RING", 8);
    if (H == GRU_H_WIDE) {
        MMS_REQUIRE(ring > 0, "gru_recur_bwd: GRU_BWD_RING=0 selects the register-ring backward, which has no hidden size %d kernel", H);
        MMS_REQUIRE(bwd_ring_ok(prm, ndirs),
                    "gru_recur_bwd: at hidden size %d stash / hs / dout must be 16-byte aligned with strides that are multiples of 4 floats", H);
    }
    if (ring > 0 && R == 1 && bwd_ring_ok(prm, ndirs)) {
        // MMS_GRU_BWD_EXCLUSIVE_KB (experiment, default 0): reserve that much dynamic shared memory per CTA so that no
        // other kernel's CTAs (the weight-gradient GEMMs of the side streams) can share an SM with a recurrence CTA
        const int excl = option_get("GRU_BWD_EXCLUSIVE_KB", 0);
        size_t dyn = 0;
        if (excl > 0) {
            dyn = (size_t)(excl > 200 ? 200 : excl) * 1024;
            static PerDeviceOnce attr_once;
            if (attr_once.need()) {
                MMS_CUDA(cudaFuncSetAttribute(gru_bwd_ring_kernel<H, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
                MMS_CUDA(cudaFuncSetAttribute(gru_bwd_ring_kernel<H, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
               
            }
        }
        MMS_PROF_BEGIN(st);
        auto r8 = gru_bwd_ring_kernel<H, 8>;
        auto r4 = gru_bwd_ring_kernel<H, 4>;
        if (ring >= 8) MMS_LAUNCH(r8, grid, dim3(2 * H), dyn, st, prm);
        else MMS_LAUNCH(r4, grid, dim3(2 * H), dyn, st, prm);
        MMS_LAUNCH_CHECK("gru_bwd_ring_kernel");
        return MMS_OK;
    }
    if constexpr (H != GRU_H_WIDE) {
        MMS_PROF_BEGIN(st);
        if (R == 1) gru_bwd_kernel<H, 1><<<grid, 2 * H, 0, st>>>(prm);
        else if (R == 2) gru_bwd_kernel<H, 2><<<grid, 2 * H, 0, st>>>(prm);
        else gru_bwd_kernel<H, 4><<<grid, 2 * H, 0, st>>>(prm);
        MMS_LAUNCH_CHECK("gru_bwd_kernel");
    }
    return MMS_OK;
}

int launch_gru_fwd(const mms_gru_dir_fwd* dirs, int ndirs, int B, int H, float p, uint64_t seed, uint64_t offset,
                   const int64_t* offset_dev, cudaStream_t st) {
    MMS_REQUIRE(ndirs >= 1 && ndirs <= GRU_MAX_DIRS && B > 0, "gru_recur_fwd: bad direction count / batch");
    MMS_REQUIRE(H == 32 || H == 64 || H == GRU_H_WIDE, "gru_recur_fwd: hidden size %d not supported (32, 64 or 128)", H);
    GruFwdParams prm;
    for (int i = 0; i < ndirs; ++i) {
        prm.dir[i] = dirs[i];
        MMS_REQUIRE(dirs[i].gi && dirs[i].w_hh && dirs[i].b_hh && dirs[i].hs && dirs[i].nsteps >= 1, "gru_recur_fwd: null pointer / no steps");
        MMS_REQUIRE(!dirs[i].hs_drop, "gru_recur_fwd: hs_drop is no longer written by the recurrence; use mms_dropout_apply");
        MMS_REQUIRE((reinterpret_cast<uintptr_t>(dirs[i].gi) & 15) == 0 && dirs[i].gi_bs % 4 == 0 && dirs[i].gi_ts % 4 == 0,
                    "gru_recur_fwd: gi must be 16-byte aligned with strides that are multiples of 4 floats");
    }
    for (int i = ndirs; i < GRU_MAX_DIRS; ++i) prm.dir[i] = dirs[0];
    prm.B = B; prm.p = p; prm.seed = seed; prm.offset = offset; prm.offset_dev = offset_dev;
    if (H == GRU_H_WIDE) return gru_fwd_dispatch<GRU_H_WIDE>(prm, ndirs, st);
    return H == 64 ? gru_fwd_dispatch<64>(prm, ndirs, st) : gru_fwd_dispatch<32>(prm, ndirs, st);
}

int launch_gru_bwd(const mms_gru_dir_bwd* dirs, int ndirs, int B, int H, float p, uint64_t seed, uint64_t offset,
                   const int64_t* offset_dev, cudaStream_t st) {
    MMS_REQUIRE(ndirs >= 1 && ndirs <= GRU_MAX_DIRS && B > 0, "gru_recur_bwd: bad direction count / batch");
    MMS_REQUIRE(H == 32 || H == 64 || H == GRU_H_WIDE, "gru_recur_bwd: hidden size %d not supported (32, 64 or 128)", H);
    GruBwdParams prm;
    for (int i = 0; i < ndirs; ++i) {
        prm.dir[i] = dirs[i];
        MMS_REQUIRE(dirs[i].w_hh && dirs[i].stash && dirs[i].hs && dirs[i].D && dirs[i].nsteps >= 1, "gru_recur_bwd: null pointer / no steps");
        MMS_REQUIRE(!dirs[i].dh_head || dirs[i].w0, "gru_recur_bwd: dh_head needs w0");
        MMS_REQUIRE(!dirs[i].drop_mask, "gru_recur_bwd: drop_mask is no longer applied by the recurrence; use mms_dropout_apply");
    }
    for (int i = ndirs; i < GRU_MAX_DIRS; ++i) prm.dir[i] = dirs[0];
    prm.B = B; prm.p = p; prm.seed = seed; prm.offset = offset; prm.offset_dev = offset_dev;
    if (H == GRU_H_WIDE) return gru_bwd_dispatch<GRU_H_WIDE>(prm, ndirs, st);
    return H == 64 ? gru_bwd_dispatch<64>(prm, ndirs, st) : gru_bwd_dispatch<32>(prm, ndirs, st);
}

}  // namespace mms

using namespace mms;

extern "C" int mms_gru_recur_fwd(const mms_gru_dir_fwd* dirs_host, int32_t ndirs, int32_t B, int32_t H, float dropout_p,
                                 uint64_t rng_seed, uint64_t rng_offset, const int64_t* rng_offset_dev, mms_stream_t stream) {
    MMS_REQUIRE(dirs_host, "gru_recur_fwd: null dirs");
    return launch_gru_fwd(dirs_host, ndirs, B, H, dropout_p, rng_seed, rng_offset, rng_offset_dev, (cudaStream_t)stream);
}
extern "C" int mms_gru_recur_bwd(const mms_gru_dir_bwd* dirs_host, int32_t ndirs, int32_t B, int32_t H, float dropout_p,
                                 uint64_t rng_seed, uint64_t rng_offset, const int64_t* rng_offset_dev, mms_stream_t stream) {
    MMS_REQUIRE(dirs_host, "gru_recur_bwd: null dirs");
    return launch_gru_bwd(dirs_host, ndirs, B, H, dropout_p, rng_seed, rng_offset, rng_offset_dev, (cudaStream_t)stream);
}
