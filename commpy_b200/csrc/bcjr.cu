// BCJR (MAP) decoding and the turbo loop on sm_100a -- replaces commpy/channelcoding/turbo.py:78-111
// (_backward_recursion), :114-158 (_forward_recursion_decoding), :163-251 (map_decode) and the iteration
// loop of :254-333 (turbo_decode).
//
// Kernel families (all compute the exact MAP of the reference, float32 instead of float64):
//   tpf::map_lin2_kernel<T,SM> the hot one (systematic compile-time trellis T, frame length a multiple of 4): PROBABILITY
//                            domain like the reference itself, one THREAD per (frame, window of 1024 steps) with a 96-step
//                            warm-up of alpha and beta over the neighbouring windows; four branch weights per step relative
//                            to the most likely (input, parity) pair; metrics rescaled every 4th step (the reference
//                            rescales every step, turbo.py:106-111,155 -- a block whose sum decays is redone per step); beta
//                            checkpointed every 8 steps in a global scratch and recomputed per segment in shared memory; in
//                            the turbo loop it writes the extrinsic L - L_int itself.  SM = step-major arrays
//                            [step][frame]: inputs staged by cp.async, the interleaver is a row index (turbo loop);
//                            otherwise frame-major rows read as 16-byte vectors (map_decode).
//   tpf::map_lin_kernel<T>   the same with per-step rescaling and separate prior / channel weights (non-systematic
//                            compile-time trellises; cross-check of map_lin2 behind CPB_OPT_BCJR_PER_STEP_SCALING).
//   tpf::map_tpf_kernel<T>   log2-domain exact max* form of the same thread mapping, scalar loads, beta of every step in
//                            global scratch (frame lengths not a multiple of 4, unaligned rows).
//   map_kernel<S>            table-driven fallback for any other rate-1/2 trellis with <= 32 states: one LANE per state,
//                            32/S frames per warp, neighbour metrics by warp shuffle, full-frame recursions (no windows),
//                            log domain:
//   gamma_t(s,u) = -((ys_t-(2cs-1))^2 + (yp_t-(2cp-1))^2) / (2 sigma^2)         turbo.py:62-76   (cs = MSB of the
//                                                                                output symbol, cp = LSB, :97-99)
//   beta_{t-1}(s) = max*_u  beta_t(ns(s,u)) + gamma_t(s,u) + u*La_t             :106-108, beta_N = 0 (:225-226)
//   alpha_t(ns)   = max*    alpha_{t-1}(s)  + gamma_t(s,u) + u*La_t             :136-138, alpha_0 = delta(s,0)
//   L_t = La_t + max*_s[alpha_{t-1}(s)+gamma_t(s,1)+beta_t(ns(s,1))] - max*_s[... u = 0 ...]     :141-146
// (log P(u) = u*La - softplus(La); the common term cancels like the reference's normalisations do).
// The turbo loop (cpb_turbo_decode) transposes the three symbol streams to step-major once and then runs 2 MAP launches per
// iteration -- decoder 2 addresses rows through the interleaver, so no data is permuted; on trellises / lengths the
// step-major kernel does not take it is 2 MAP launches + 2 row-staged interleaver launches per iteration on frame-major rows.
#include <algorithm>

#include <cstdlib>

#include "common.cuh"

using namespace cpb;

struct cpbTrellis;
const int32_t *cpb_trellis_next_dev(const cpbTrellis *t);
const int32_t *cpb_trellis_out_dev(const cpbTrellis *t);
void cpb_trellis_dims(const cpbTrellis *t, int *k, int *n, int *S);
const int32_t *cpb_trellis_pred_dev(const cpbTrellis *t);
void cpb_trellis_host_tables(const cpbTrellis *t, const int32_t **next, const int32_t **out);

namespace bcjr {

constexpr float NEG = -1.0e30f;

__device__ __forceinline__ float maxstar(float a, float b)
{
    const float m = fmaxf(a, b);
    return m + __logf(1.0f + __expf(-fabsf(a - b)));
}

// maximum over the S lanes of one frame
template <int S>
__device__ __forceinline__ float seg_max(float v)
{
#pragma unroll
    for (int o = S / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

template <int S>
__global__ void __launch_bounds__(128) map_kernel(const float *__restrict__ sys, const float *__restrict__ par,
                                                  const float *__restrict__ La, int64_t batch, int N,
                                                  const int32_t *__restrict__ next_tab, const int32_t *__restrict__ out_tab,
                                                  const int32_t *__restrict__ pred_tab, float inv2s2, int mode,
                                                  float *__restrict__ beta, float *__restrict__ L_out,
                                                  uint8_t *__restrict__ bits_out)
{
    constexpr int FPW = 32 / S;                  // frames per warp
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int s = lane % S, sub = lane / S;
    const int lane0 = sub * S;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int64_t f = warp * FPW + sub;
    const bool valid = f < batch;
    if (!valid) f = batch - 1;

    // trellis constants of this lane's state
    const int ns0 = __ldg(&next_tab[s * 2 + 0]), ns1 = __ldg(&next_tab[s * 2 + 1]);
    const int o0 = __ldg(&out_tab[s * 2 + 0]), o1 = __ldg(&out_tab[s * 2 + 1]);
    const float cs0 = (float)(2 * ((o0 >> 1) & 1) - 1), cp0 = (float)(2 * (o0 & 1) - 1);
    const float cs1 = (float)(2 * ((o1 >> 1) & 1) - 1), cp1 = (float)(2 * (o1 & 1) - 1);
    const int pa = __ldg(&pred_tab[s * 2 + 0]), pb = __ldg(&pred_tab[s * 2 + 1]);     // p | u<<8 | out<<16
    const int pa_s = pa & 0xff, pa_u = (pa >> 8) & 0xff, pa_o = (pa >> 16) & 0xff;
    const int pb_s = pb & 0xff, pb_u = (pb >> 8) & 0xff, pb_o = (pb >> 16) & 0xff;
    const float acs = (float)(2 * ((pa_o >> 1) & 1) - 1), acp = (float)(2 * (pa_o & 1) - 1);
    const float bcs = (float)(2 * ((pb_o >> 1) & 1) - 1), bcp = (float)(2 * (pb_o & 1) - 1);

    const float *fs = sys + f * N, *fp = par + f * N, *fl = La + f * N;
    float *fb = beta + f * (int64_t)(N + 1) * S;

    auto gamma = [&](float ys, float yp, float cs, float cp) {
        const float a = ys - cs, b = yp - cp;
        return -(a * a + b * b) * inv2s2;
    };

    // ---- backward recursion: beta_N = 0 for every state ----
    float bt = 0.0f;
    fb[(int64_t)N * S + s] = 0.0f;
    for (int t1 = N; t1 >= 1; t1 -= S) {             // steps t1, t1-1, ..., t1-S+1 (lane i holds step t1-i)
        const int tl = t1 - s;
        float vs = 0.f, vp = 0.f, vl = 0.f;
        if (tl >= 1) { vs = __ldg(fs + tl - 1); vp = __ldg(fp + tl - 1); vl = __ldg(fl + tl - 1); }
#pragma unroll
        for (int i = 0; i < S; ++i) {
            const int t = t1 - i;
            if (t < 1) break;                         // warp-uniform
            const float ys = __shfl_sync(FULL, vs, lane0 + i), yp = __shfl_sync(FULL, vp, lane0 + i);
            const float la = __shfl_sync(FULL, vl, lane0 + i);
            const float b0 = __shfl_sync(FULL, bt, lane0 + ns0), b1 = __shfl_sync(FULL, bt, lane0 + ns1);
            float nb = maxstar(b0 + gamma(ys, yp, cs0, cp0), b1 + gamma(ys, yp, cs1, cp1) + la);
            bt = nb - seg_max<S>(nb);                 // keep the metrics bounded (the reference divides by the sum)
            fb[(int64_t)(t - 1) * S + s] = bt;
        }
    }

    // ---- forward recursion + a-posteriori LLR ----
    float at = (s == 0) ? 0.0f : NEG;                 // alpha_0 = delta(s, 0), turbo.py:220-221
    for (int t0 = 1; t0 <= N; t0 += S) {              // steps t0 .. t0+S-1 (lane i holds step t0+i)
        const int tl = t0 + s;
        float vs = 0.f, vp = 0.f, vl = 0.f;
        if (tl <= N) { vs = __ldg(fs + tl - 1); vp = __ldg(fp + tl - 1); vl = __ldg(fl + tl - 1); }
        float keep = 0.0f;
#pragma unroll
        for (int i = 0; i < S; ++i) {
            const int t = t0 + i;
            if (t > N) break;
            const float ys = __shfl_sync(FULL, vs, lane0 + i), yp = __shfl_sync(FULL, vp, lane0 + i);
            const float la = __shfl_sync(FULL, vl, lane0 + i);
            const float bown = fb[(int64_t)t * S + s];
            const float b0 = __shfl_sync(FULL, bown, lane0 + ns0), b1 = __shfl_sync(FULL, bown, lane0 + ns1);
            float a0 = at + gamma(ys, yp, cs0, cp0) + b0;        // APP terms exclude the prior (:141-143)
            float a1 = at + gamma(ys, yp, cs1, cp1) + b1;
#pragma unroll
            for (int o = S / 2; o > 0; o >>= 1) {
                a0 = maxstar(a0, __shfl_xor_sync(FULL, a0, o));
                a1 = maxstar(a1, __shfl_xor_sync(FULL, a1, o));
            }
            const float L = la + (a1 - a0);                       // :145
            if (i == s) keep = L;
            const float xa = __shfl_sync(FULL, at, lane0 + pa_s), xb = __shfl_sync(FULL, at, lane0 + pb_s);
            float na = maxstar(xa + gamma(ys, yp, acs, acp) + (pa_u ? la : 0.0f),
                               xb + gamma(ys, yp, bcs, bcp) + (pb_u ? la : 0.0f));
            // a state whose predecessors are both unreachable keeps the sentinel instead of drifting
            at = fmaxf(na - seg_max<S>(na), NEG);
        }
        if (valid && tl <= N) {
            L_out[f * N + tl - 1] = keep;
            if (bits_out) bits_out[f * N + tl - 1] = (uint8_t)((mode == 1 && keep > 0.0f) ? 1 : 0);   // :148-152
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Register-resident MAP kernel: ONE THREAD per (frame, window), all S <= 8 state metrics in registers, the
// trellis baked in at compile time (NEXT/OUT pack Trellis.next_state_table / output_table, 3 and 2 bits per
// entry), so every table look-up is a register name.  Metrics live in the log2 domain: with a = ys*log2e/s^2,
// b = yp*log2e/s^2 the branch metric of output (cs,cp) is +-a +-b (terms common to all branches of a step
// cancel in every max* and in the LLR), max*(x,y) = max + lg2(1 + ex2(-|x-y|)) is two raw MUFU ops.
// A frame longer than 1536 steps is cut into windows of 1024 steps; alpha starts 96 steps before its window and
// beta 96 steps after it from uniform metrics (the true boundary values where the window touches the frame
// ends).  SURVEY.md section 7-5 measured this warm-up against the reference's full-frame recursion: <= 3.4e-7
// on the LLRs, i.e. inside fp32 round-off; the split depends only on N, never on the batch, so a frame decodes
// identically whatever it is batched with.
// ------------------------------------------------------------------------------------------------
namespace tpf {

constexpr float NEGM = -1.0e30f;
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;
constexpr int WIN = 1024, WARM = 96;

__device__ __forceinline__ float ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float maxstar2(float x, float y)
{
    return fmaxf(x, y) + lg2(1.0f + ex2(-fabsf(x - y)));
}

template <int S_, unsigned long long NEXT_, unsigned int OUT_>
struct CT {
    static constexpr int S = S_;
    __host__ __device__ static constexpr int ns(int s, int u) { return (int)((NEXT_ >> (3 * (2 * s + u))) & 7ull); }
    __host__ __device__ static constexpr int out(int s, int u) { return (int)((OUT_ >> (2 * (2 * s + u))) & 3u); }
    // idx-th edge (packed 2*s+u) entering state n, in (s asc, u asc) order
    __host__ __device__ static constexpr int pred(int n, int idx)
    {
        int c = 0;
        for (int e = 0; e < 2 * S_; ++e)
            if (ns(e >> 1, e & 1) == n) { if (c == idx) return e; ++c; }
        return -1;
    }
    __host__ __device__ static constexpr bool valid()
    {
        for (int n = 0; n < S_; ++n) { if (pred(n, 1) < 0 || pred(n, 2) >= 0) return false; }
        return true;
    }
};

struct Params {
    const float *sys, *par, *La;
    int64_t batch, bp;           // frames, frames padded to a multiple of 32
    int N, nwin, win;            // frame length, windows per frame, steps per window
    float c;                     // log2(e) / sigma^2
    int mode;
    float *beta;                 // [(tloc*S + s) * NT + thread]
    int64_t NT;
    float *L_out;
    uint8_t *bits_out;
    int ext;                     // map_lin_kernel only: L_out receives L - La (the extrinsic turbo_decode forms, turbo.py:318,328)
    // step-major arrays (map_lin2_kernel<T, true>, the turbo loop): element (step t, frame f) at [row(t) * pitch + f];
    // sys, La, L_out and bits_out use row(t) = rmap ? rmap[t] : t (the interleaver, interleavers.py:13-47), par uses row t
    int64_t pitch;
    const int32_t *rmap;
};

// the log2-domain kernel for frame lengths that are not a multiple of 4 or rows that are not 16-byte aligned: scalar
// loads, the beta of every step of the window in a global scratch
template <class T>
__global__ void __launch_bounds__(128) map_tpf_kernel(const Params p)
{
    // steps per group (one: scalar loads).  The one-step group loops are kept on purpose: written without them, the kernel
    // compiles to a different instruction schedule from the one it has been tested and measured with.
    constexpr int G = 1;
    constexpr int S = T::S;
    static_assert(T::valid(), "every state needs exactly two incoming edges");
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= p.NT) return;
    const int w = (int)(g / p.bp);
    const int64_t f = g - (int64_t)w * p.bp;
    if (f >= p.batch) return;
    const int N = p.N;
    const int lo = w * p.win, hi = min(N, lo + p.win);       // this thread emits steps lo+1 .. hi
    const float *fs = p.sys + f * N, *fp = p.par + f * N, *fl = p.La + f * N;
    float *bcol = p.beta + g;

    float A[S], B[S];
    auto branch = [&](float ys, float yp, float (&gm)[4]) {
        const float a = ys * p.c, b = yp * p.c;
        gm[0] = -a - b; gm[1] = b - a; gm[2] = a - b; gm[3] = a + b;      // output symbol (cs,cp): MSB = systematic
    };
    auto load = [&](const float *q, int e0, float (&v)[G]) { v[0] = __ldg(q + e0); };

    // ---- backward: beta_t for t = tb .. lo+1, stored for t <= hi (inputs prefetched one group ahead)
    {
        const int tb = min(N, hi + WARM);
#pragma unroll
        for (int s = 0; s < S; ++s) B[s] = 0.0f;                          // beta_N = 1 / uniform warm-up start
        float ns_[G], np_[G], nl_[G];
        load(fs, tb - G, ns_); load(fp, tb - G, np_); load(fl, tb - G, nl_);
        for (int e1 = tb; e1 > lo; e1 -= G) {                             // steps e1, e1-1, .., e1-G+1
            float vs[G], vp[G], vl[G];
#pragma unroll
            for (int i = 0; i < G; ++i) { vs[i] = ns_[i]; vp[i] = np_[i]; vl[i] = nl_[i]; }
            if (e1 - G > lo) { load(fs, e1 - 2 * G, ns_); load(fp, e1 - 2 * G, np_); load(fl, e1 - 2 * G, nl_); }
#pragma unroll
            for (int i = G - 1; i >= 0; --i) {
                const int t = e1 - (G - 1 - i);
                if (t <= hi) {
#pragma unroll
                    for (int s = 0; s < S; ++s) bcol[((int64_t)(t - lo - 1) * S + s) * p.NT] = B[s];
                }
                float gm[4];
                branch(vs[i], vp[i], gm);
                const float la = vl[i] * LOG2E;
                float Bn[S];
#pragma unroll
                for (int s = 0; s < S; ++s)
                    Bn[s] = maxstar2(B[T::ns(s, 0)] + gm[T::out(s, 0)], B[T::ns(s, 1)] + gm[T::out(s, 1)] + la);
                if ((t & 3) == 1) {                                       // renormalise every 4th step
                    float m = Bn[0];
#pragma unroll
                    for (int s = 1; s < S; ++s) m = fmaxf(m, Bn[s]);
#pragma unroll
                    for (int s = 0; s < S; ++s) Bn[s] -= m;
                }
#pragma unroll
                for (int s = 0; s < S; ++s) B[s] = Bn[s];
            }
        }
    }
    // ---- forward: alpha from ta, LLRs for t = lo+1 .. hi (inputs one group ahead, beta one step ahead)
    {
        const int ta = max(0, lo - WARM);
#pragma unroll
        for (int s = 0; s < S; ++s) A[s] = (ta == 0 && s != 0) ? NEGM : 0.0f;   // alpha_0 = delta(s,0) / uniform
        auto load_beta = [&](int t, float (&b)[S]) {
            if (t > lo && t <= hi) {
#pragma unroll
                for (int s = 0; s < S; ++s) b[s] = bcol[((int64_t)(t - lo - 1) * S + s) * p.NT];
            }
        };
        float bnext[S];
#pragma unroll
        for (int s = 0; s < S; ++s) bnext[s] = 0.0f;
        load_beta(ta + 1, bnext);
        float ns_[G], np_[G], nl_[G];
        load(fs, ta, ns_); load(fp, ta, np_); load(fl, ta, nl_);
        for (int e0 = ta; e0 < hi; e0 += G) {                              // steps e0+1 .. e0+G
            float vs[G], vp[G], vl[G];
#pragma unroll
            for (int i = 0; i < G; ++i) { vs[i] = ns_[i]; vp[i] = np_[i]; vl[i] = nl_[i]; }
            if (e0 + G < hi) { load(fs, e0 + G, ns_); load(fp, e0 + G, np_); load(fl, e0 + G, nl_); }
            float Lv[G];
#pragma unroll
            for (int i = 0; i < G; ++i) {
                const int t = e0 + 1 + i;
                float bt[S];
#pragma unroll
                for (int s = 0; s < S; ++s) bt[s] = bnext[s];
                load_beta(t + 1, bnext);
                float gm[4];
                branch(vs[i], vp[i], gm);
                const float la = vl[i] * LOG2E;
                float tx[2 * S];
#pragma unroll
                for (int e = 0; e < 2 * S; ++e) tx[e] = A[e >> 1] + gm[T::out(e >> 1, e & 1)];
                Lv[i] = 0.0f;
                if (t > lo) {
                    float x0[S], x1[S];
#pragma unroll
                    for (int s = 0; s < S; ++s) {
                        x0[s] = tx[2 * s] + bt[T::ns(s, 0)];               // APP terms exclude the prior (turbo.py:141-143)
                        x1[s] = tx[2 * s + 1] + bt[T::ns(s, 1)];
                    }
                    float m0 = x0[0], m1 = x1[0];
#pragma unroll
                    for (int s = 1; s < S; ++s) { m0 = fmaxf(m0, x0[s]); m1 = fmaxf(m1, x1[s]); }
                    float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
                    for (int s = 0; s < S; ++s) { s0 += ex2(x0[s] - m0); s1 += ex2(x1[s] - m1); }
                    Lv[i] = vl[i] + LN2 * ((m1 + lg2(s1)) - (m0 + lg2(s0)));   // turbo.py:145
                }
                float An[S];
#pragma unroll
                for (int n = 0; n < S; ++n) {
                    const int ea = T::pred(n, 0), eb = T::pred(n, 1);
                    An[n] = maxstar2(tx[ea] + ((ea & 1) ? la : 0.0f), tx[eb] + ((eb & 1) ? la : 0.0f));
                }
                if ((t & 3) == 0) {
                    float m = An[0];
#pragma unroll
                    for (int s = 1; s < S; ++s) m = fmaxf(m, An[s]);
#pragma unroll
                    for (int s = 0; s < S; ++s) An[s] = fmaxf(An[s] - m, NEGM);
                }
#pragma unroll
                for (int s = 0; s < S; ++s) A[s] = An[s];
            }
            if (e0 >= lo) {
                p.L_out[f * N + e0] = Lv[0];
                if (p.bits_out) p.bits_out[f * N + e0] = (uint8_t)((p.mode == 1 && Lv[0] > 0.0f) ? 1 : 0);   // :148-152
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Probability-domain variant (what actually runs for N % 4 == 0): the log-domain kernel above spends 66 MUFU
// operations per trellis step (ex2 + lg2 per max*) and is bound by the 16-lane XU pipe.  The reference itself
// works with probabilities renormalised every step (turbo.py:106-111, :155); doing the same in fp32 needs only
// multiplies and adds for the recursions:
//   branch weight of output symbol (cs, cp), relative to the best symbol of the step (all weights <= 1, no
//   overflow):  w = [cs opposes ys ? 2^(-2|a|) : 1] * [cp opposes yp ? 2^(-2|b|) : 1],  a = ys log2e/s^2, b = yp log2e/s^2
//   prior odds P(1)/P(0) = e^La, also relative to the larger:  (p0, p1) = La > 0 ? (2^(-La log2e), 1) : (1, 2^(La log2e))
//   beta_{t-1}(s) = sum_u p_u w(s,u) beta_t(ns(s,u)),  alpha_t(ns) += p_u w(s,u) alpha_{t-1}(s),  both rescaled to sum 1
//   L_t = La + ln( sum_s alpha w(s,1) beta / sum_s alpha w(s,0) beta )
// i.e. 2 + 1 ex2, 3 reciprocals and 2 lg2 per step instead of 66 MUFU ops.  |a|, |b|, |La log2e| are clamped to 60
// so nothing reaches the fp32 exponent limits; the clamp only acts where |LLR| > ~80.
// Beta is written to HBM only every CK-th step.  The forward sweep then works segment by segment: reload the CK steps of
// inputs into shared memory, recompute the segment's beta backwards from its checkpoint (same operations in the same
// order as the first sweep, so the same values), then run alpha / the a-posteriori LLRs forwards.  This trades +1 beta
// recursion per step for 8x less beta traffic: map_tpf_kernel, which stores the beta of every step, moved 4.7 GB per pass
// for a batch of 8192 x 6144 (3.2 GB of it beta), i.e. it was HBM bound on non-algorithmic bytes
// (profiles/r01_other_kernels_ncu.md).
// Shared memory per thread: CK*(S+3) floats, thread-private columns [slot][thread] (conflict free).
// ------------------------------------------------------------------------------------------------
constexpr int CK = 8;

__device__ __forceinline__ float rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

template <class T>
__global__ void __launch_bounds__(128) map_lin_kernel(const Params p)
{
    constexpr int S = T::S;
    constexpr int G = 4;
    extern __shared__ float smem_f[];
    const int tid = threadIdx.x, bd = blockDim.x;
    float *sb = smem_f;                         // [CK][S][bd]
    float *si = smem_f + CK * S * bd;           // [CK][3][bd]
    const int64_t g = (int64_t)blockIdx.x * bd + tid;
    if (g >= p.NT) return;
    const int w = (int)(g / p.bp);
    const int64_t f = g - (int64_t)w * p.bp;
    if (f >= p.batch) return;
    const int N = p.N;
    const int lo = w * p.win, hi = min(N, lo + p.win);
    const float *fs = p.sys + f * N, *fp = p.par + f * N, *fl = p.La + f * N;
    float *ck = p.beta + g;

    // weights of the four output symbols (index o = cs<<1 | cp with cs/cp = 1 for +1) and the two prior factors
    auto weights = [&](float ys, float yp, float la_raw, float (&wt)[4], float &p0, float &p1) {
        const float a = fminf(fmaxf(ys * p.c, -60.0f), 60.0f), b = fminf(fmaxf(yp * p.c, -60.0f), 60.0f);
        const float ea = ex2(-2.0f * fabsf(a)), eb = ex2(-2.0f * fabsf(b));
        const float s1 = (a >= 0.0f) ? 1.0f : ea, s0 = (a >= 0.0f) ? ea : 1.0f;      // systematic bit +1 / -1
        const float q1 = (b >= 0.0f) ? 1.0f : eb, q0 = (b >= 0.0f) ? eb : 1.0f;      // parity bit +1 / -1
        wt[0] = s0 * q0; wt[1] = s0 * q1; wt[2] = s1 * q0; wt[3] = s1 * q1;
        const float l = fminf(fmaxf(la_raw * LOG2E, -60.0f), 60.0f);
        const float el = ex2(-fabsf(l));
        p0 = (l > 0.0f) ? el : 1.0f;
        p1 = (l > 0.0f) ? 1.0f : el;
    };
    auto normalise = [&](float (&v)[S]) {
        float sum = v[0];
#pragma unroll
        for (int s = 1; s < S; ++s) sum += v[s];
        const float r = rcp(fmaxf(sum, 1.0e-37f));
#pragma unroll
        for (int s = 0; s < S; ++s) v[s] *= r;
    };
    auto beta_step = [&](float (&B)[S], float ys, float yp, float la_raw) {           // beta_t -> beta_{t-1}
        float wt[4], p0, p1;
        weights(ys, yp, la_raw, wt, p0, p1);
        float w0[4], w1[4];
#pragma unroll
        for (int o = 0; o < 4; ++o) { w0[o] = wt[o] * p0; w1[o] = wt[o] * p1; }
        float Bn[S];
#pragma unroll
        for (int s = 0; s < S; ++s)
            Bn[s] = w0[T::out(s, 0)] * B[T::ns(s, 0)] + w1[T::out(s, 1)] * B[T::ns(s, 1)];      // turbo.py:106-108
        normalise(Bn);                                                                          // :110-111
#pragma unroll
        for (int s = 0; s < S; ++s) B[s] = Bn[s];
    };
    auto ld4 = [&](const float *q, int e0, float (&v)[G]) {
        const float4 t = __ldg(reinterpret_cast<const float4 *>(q + e0));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    };

    // ---- backward sweep with checkpoints
    {
        float B[S];
        const int tb = min(N, hi + WARM);
#pragma unroll
        for (int s = 0; s < S; ++s) B[s] = 1.0f / S;                      // beta_N = 1 for all states (:225-226), scale free
        // inputs are fetched two groups (8 steps) ahead of their use: with ~10 warps per SM a DRAM round trip is longer
        // than one group of beta steps
        float ns_[G], np_[G], nl_[G], ms_[G], mp_[G], ml_[G];
        ld4(fs, tb - G, ns_); ld4(fp, tb - G, np_); ld4(fl, tb - G, nl_);
        if (tb - G > lo) { ld4(fs, tb - 2 * G, ms_); ld4(fp, tb - 2 * G, mp_); ld4(fl, tb - 2 * G, ml_); }
        for (int e1 = tb; e1 > lo; e1 -= G) {
            float vs[G], vp[G], vl[G];
#pragma unroll
            for (int i = 0; i < G; ++i) {
                vs[i] = ns_[i]; vp[i] = np_[i]; vl[i] = nl_[i];
                ns_[i] = ms_[i]; np_[i] = mp_[i]; nl_[i] = ml_[i];
            }
            if (e1 - 2 * G > lo) { ld4(fs, e1 - 3 * G, ms_); ld4(fp, e1 - 3 * G, mp_); ld4(fl, e1 - 3 * G, ml_); }
#pragma unroll
            for (int i = G - 1; i >= 0; --i) {
                const int t = e1 - (G - 1 - i);
                if (t <= hi && (((t - lo) % CK) == 0 || t == hi)) {
                    const int j = (t - lo + CK - 1) / CK - 1;
#pragma unroll
                    for (int s = 0; s < S; ++s) ck[((int64_t)j * S + s) * p.NT] = B[s];
                }
                beta_step(B, vs[i], vp[i], vl[i]);
            }
        }
    }
    // ---- forward sweep
    float A[S];
    const int ta = max(0, lo - WARM);
#pragma unroll
    for (int s = 0; s < S; ++s) A[s] = (ta == 0) ? ((s == 0) ? 1.0f : 0.0f) : (1.0f / S);    // alpha_0 = delta(s,0), :220-221
    auto alpha_step = [&](float ys, float yp, float la_raw, const float *bt, bool emit, float &Lout) {
        float wt[4], p0, p1;
        weights(ys, yp, la_raw, wt, p0, p1);
        float tx[2 * S];
#pragma unroll
        for (int e = 0; e < 2 * S; ++e) tx[e] = A[e >> 1] * wt[T::out(e >> 1, e & 1)];
        if (emit) {
            float a0 = 0.0f, a1 = 0.0f;
#pragma unroll
            for (int s = 0; s < S; ++s) {                       // the a-posteriori sums leave the prior out (:141-143)
                a0 += tx[2 * s] * bt[T::ns(s, 0) * bd];
                a1 += tx[2 * s + 1] * bt[T::ns(s, 1) * bd];
            }
            Lout = la_raw + LN2 * (lg2(fmaxf(a1, 1.0e-37f)) - lg2(fmaxf(a0, 1.0e-37f)));       // :145
        }
        float An[S];
#pragma unroll
        for (int n = 0; n < S; ++n) {
            const int ea = T::pred(n, 0), eb = T::pred(n, 1);
            An[n] = tx[ea] * ((ea & 1) ? p1 : p0) + tx[eb] * ((eb & 1) ? p1 : p0);             // :136-138
        }
        normalise(An);                                                                          // :155
#pragma unroll
        for (int s = 0; s < S; ++s) A[s] = An[s];
    };
    for (int e0 = ta; e0 < lo; e0 += G) {                       // warm-up (no LLRs, no beta)
        float vs[G], vp[G], vl[G];
        ld4(fs, e0, vs); ld4(fp, e0, vp); ld4(fl, e0, vl);
        float dummy;
#pragma unroll
        for (int i = 0; i < G; ++i) alpha_step(vs[i], vp[i], vl[i], nullptr, false, dummy);
    }
    // the inputs and the beta checkpoint of a segment are fetched while the previous segment is being processed
    static_assert(CK == 2 * G, "segment = two vector groups");
    float xin[2][3][G], xck[S];
    auto fetch_segment = [&](int s0, int j) {
        const int ns = min(CK, hi - s0);
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (h * G < ns) { ld4(fs, s0 + h * G, xin[h][0]); ld4(fp, s0 + h * G, xin[h][1]); ld4(fl, s0 + h * G, xin[h][2]); }
#pragma unroll
        for (int s = 0; s < S; ++s) xck[s] = ck[((int64_t)j * S + s) * p.NT];
    };
    if (lo < hi) fetch_segment(lo, 0);
    for (int s0 = lo, j = 0; s0 < hi; s0 += CK, ++j) {
        const int ns = min(CK, hi - s0);                        // a multiple of 4
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (h * G < ns) {
#pragma unroll
                for (int i = 0; i < G; ++i) {
                    si[((h * G + i) * 3 + 0) * bd + tid] = xin[h][0][i];
                    si[((h * G + i) * 3 + 1) * bd + tid] = xin[h][1][i];
                    si[((h * G + i) * 3 + 2) * bd + tid] = xin[h][2][i];
                }
            }
        }
        float B[S];
#pragma unroll
        for (int s = 0; s < S; ++s) B[s] = xck[s];
        if (s0 + CK < hi) fetch_segment(s0 + CK, j + 1);
        for (int i = ns - 1; i >= 0; --i) {
#pragma unroll
            for (int s = 0; s < S; ++s) sb[(i * S + s) * bd + tid] = B[s];          // beta_{s0+1+i}
            beta_step(B, si[(i * 3 + 0) * bd + tid], si[(i * 3 + 1) * bd + tid], si[(i * 3 + 2) * bd + tid]);
        }
        for (int q = 0; q < ns; q += G) {
            float Lv[G];
#pragma unroll
            for (int i = 0; i < G; ++i) {
                const int k = q + i;
                alpha_step(si[(k * 3 + 0) * bd + tid], si[(k * 3 + 1) * bd + tid], si[(k * 3 + 2) * bd + tid],
                           sb + (k * S) * bd + tid, true, Lv[i]);
            }
            const int e0 = s0 + q;
            if (p.ext)
                *reinterpret_cast<float4 *>(p.L_out + f * N + e0) =
                    make_float4(Lv[0] - si[((q + 0) * 3 + 2) * bd + tid], Lv[1] - si[((q + 1) * 3 + 2) * bd + tid],
                                Lv[2] - si[((q + 2) * 3 + 2) * bd + tid], Lv[3] - si[((q + 3) * 3 + 2) * bd + tid]);
            else
                *reinterpret_cast<float4 *>(p.L_out + f * N + e0) = make_float4(Lv[0], Lv[1], Lv[2], Lv[3]);
            if (p.bits_out) {
                uchar4 b;
                b.x = (p.mode == 1 && Lv[0] > 0.0f); b.y = (p.mode == 1 && Lv[1] > 0.0f);
                b.z = (p.mode == 1 && Lv[2] > 0.0f); b.w = (p.mode == 1 && Lv[3] > 0.0f);
                *reinterpret_cast<uchar4 *>(p.bits_out + f * N + e0) = b;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Block-normalised form of map_lin_kernel for SYSTEMATIC trellises (output MSB = input bit: every 'rsc' Trellis and the
// config-3 code) -- the same thread mapping, windows, checkpoints and prefetching, ~40 % fewer instructions per step:
//   * prior, systematic and parity observation are folded into FOUR weights per step, g[u][cp] = 2^-(what opposes the best
//     (u, cp)), computed once per sweep (2 ex2); the forward sweep keeps them in shared memory for the beta
//     recomputation AND the alpha / a-posteriori step (map_lin_kernel evaluated its 3 ex2 three times per step);
//   * the metrics are rescaled every FOURTH step instead of every step.  Scaling is arbitrary in exact arithmetic
//     (turbo.py:110-111,155 divide by the sum only to stay in range), and fp32 has the range for 4 steps of typical decay;
//     a block whose metric sum falls below 2^-20 is redone with per-step scaling from the saved metrics, so a run of
//     strongly contradicted observations (weights down to 2^-300 per step) cannot underflow;
//   * the a-posteriori sums include the prior (one multiply per edge less); L = La + ln2 (lg2 a1 - lg2 a0 - l), with l the
//     clamped log2 prior odds that went into the weights.
// ------------------------------------------------------------------------------------------------
template <class T>
__host__ __device__ constexpr bool systematic()
{
    for (int s = 0; s < T::S; ++s)
        for (int u = 0; u < 2; ++u)
            if ((T::out(s, u) >> 1) != u) return false;
    return true;
}

constexpr float RESCALE_FLOOR = 9.5367431640625e-07f;      // 2^-20
constexpr int LIN2_MIN_CTAS = 12;  // __launch_bounds__ minimum CTAs (= warps) per SM of map_lin2_kernel: <= 168 registers, three
                                   // warps per scheduler; the 1,536 warps of a config-3 pass (8,192 x 6 windows) are one wave
template <class T, bool SM>      // SM: step-major arrays (Params::pitch / rmap)
__global__ void __launch_bounds__(32, LIN2_MIN_CTAS) map_lin2_kernel(const Params p)
{
    constexpr int S = T::S;
    constexpr int G = 4;
    constexpr int SV = S / 4;                   // float4 words per metric vector
    static_assert(S % 4 == 0 && systematic<T>(), "systematic trellis with 4 or 8 states");
    extern __shared__ float4 smem_v[];
    constexpr int bd = 32;                      // one warp per CTA (launch<T>): every shared-memory offset is an immediate
    const int tid = threadIdx.x;
    float4 *sb = smem_v;                        // [CK][SV][bd]  beta of the current segment
    float4 *sg = smem_v + CK * SV * bd;         // [CK][bd]      the four branch weights of a step
    float *sl = reinterpret_cast<float *>(sg + CK * bd);   // [CK][bd]  L_int of a step
    const int64_t g = (int64_t)blockIdx.x * bd + tid;
    if (g >= p.NT) return;
    const int w = (int)(g / p.bp);
    const int64_t f = g - (int64_t)w * p.bp;
    if (f >= p.batch) return;
    const int N = p.N;
    const int lo = w * p.win, hi = min(N, lo + p.win);
    const float *fs = p.sys + f * N, *fp = p.par + f * N, *fl = p.La + f * N;
    float *ck = p.beta + g;
    const float c2 = 2.0f * p.c;
    const uint32_t NT32 = (uint32_t)p.NT;       // checkpoint (segment j, state s) at ck[(j S + s) NT]: 32-bit offsets (launch_map checks)

    // weights of the four (u, cp) pairs relative to the most likely pair: index o = u << 1 | cp
    auto weights = [&](float ys, float yp, float la_raw) -> float4 {
        // (no clamp on the channel terms: ex2 of a large negative number is 0, an infinite symbol gives weights (1, 0),
        // and the clamped prior keeps infinity - infinity out)
        const float l = fminf(fmaxf(la_raw * LOG2E, -60.0f), 60.0f);
        const float lu = fmaf(ys, c2, l);                                  // log2 odds of u = 1: channel + prior
        const float lb = yp * c2;                                          // log2 odds of cp = 1
        const float eu = ex2(-fabsf(lu)), eb = ex2(-fabsf(lb));
        const float u1 = (lu >= 0.0f) ? 1.0f : eu, u0 = (lu >= 0.0f) ? eu : 1.0f;
        const float q1 = (lb >= 0.0f) ? 1.0f : eb, q0 = (lb >= 0.0f) ? eb : 1.0f;
        return make_float4(u0 * q0, u0 * q1, u1 * q0, u1 * q1);
    };
    auto pick = [](const float4 &v, int o) -> float { return o == 0 ? v.x : (o == 1 ? v.y : (o == 2 ? v.z : v.w)); };
    auto total = [](const float (&v)[S]) {              // pairwise: three dependent adds instead of seven
        float t[S];
#pragma unroll
        for (int s = 0; s < S; ++s) t[s] = v[s];
#pragma unroll
        for (int w = S / 2; w >= 1; w >>= 1)
#pragma unroll
            for (int s = 0; s < w; ++s) t[s] += t[s + w];
        return t[0];
    };
    auto scale = [](float (&v)[S], float sum) {
        const float r = rcp(fmaxf(sum, 1.0e-37f));
#pragma unroll
        for (int s = 0; s < S; ++s) v[s] *= r;
    };
    auto beta_raw = [&](float (&B)[S], const float4 &gw) {                  // beta_t -> beta_{t-1}, turbo.py:106-108
        float Bn[S];
#pragma unroll
        for (int s = 0; s < S; ++s)
            Bn[s] = pick(gw, T::out(s, 0)) * B[T::ns(s, 0)] + pick(gw, T::out(s, 1)) * B[T::ns(s, 1)];
#pragma unroll
        for (int s = 0; s < S; ++s) B[s] = Bn[s];
    };
    // the rows of steps e0+1 .. e0+4 in the step-major arrays
    auto rows4 = [&](int e0, int (&r)[G]) {
        if (p.rmap) {
            const int4 q = __ldg(reinterpret_cast<const int4 *>(p.rmap + e0));
            r[0] = q.x; r[1] = q.y; r[2] = q.z; r[3] = q.w;
        } else {
#pragma unroll
            for (int i = 0; i < G; ++i) r[i] = e0 + i;
        }
    };
    // inputs of steps e0+1 .. e0+4 (0-based elements e0 .. e0+3)
    auto ld3 = [&](int e0, float (&vs)[G], float (&vp)[G], float (&vl)[G]) {
        if (SM) {
            int r[G];
            rows4(e0, r);
#pragma unroll
            for (int i = 0; i < G; ++i) {
                vs[i] = __ldg(p.sys + (int64_t)r[i] * p.pitch + f);
                vp[i] = __ldg(p.par + (int64_t)(e0 + i) * p.pitch + f);
                vl[i] = __ldg(p.La + (int64_t)r[i] * p.pitch + f);
            }
        } else {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(fs + e0));
            const float4 b = __ldg(reinterpret_cast<const float4 *>(fp + e0));
            const float4 c = __ldg(reinterpret_cast<const float4 *>(fl + e0));
            vs[0] = a.x; vs[1] = a.y; vs[2] = a.z; vs[3] = a.w;
            vp[0] = b.x; vp[1] = b.y; vp[2] = b.z; vp[3] = b.w;
            vl[0] = c.x; vl[1] = c.y; vl[2] = c.z; vl[3] = c.w;
        }
    };
    // ---- step-major input staging: cp.async straight into shared memory, completion by cp.async groups.  (Register
    // prefetching does not survive ptxas here: the 12 scalar loads of a group all land on one scoreboard, so the first use
    // of group n also waited for the loads of group n+1 issued a moment before -- a quarter of all warp samples.)
    // Ring of RB groups in the beta / weight area (idle during the backward sweep and the alpha warm-up); a slot holds the
    // 12 floats of a group (sys, par, L_int of 4 steps), float k of slot q at ring[(q * 12 + k) * bd + tid].
    constexpr int RB = (CK * (S + 5) / 12 >= 8) ? 8 : CK * (S + 5) / 12;          // 8 groups (6 for 4 states)
    float *ring = reinterpret_cast<float *>(smem_v);
    float *segbuf = ring + (CK * SV * 4 + CK * 4 + CK) * bd;          // forward sweep: inputs + checkpoint of the NEXT segment
    const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring) + 4u * tid;
    const uint32_t seg_s = (uint32_t)__cvta_generic_to_shared(segbuf) + 4u * tid;
    auto cp4 = [](uint32_t dst, const float *src) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
    };
    auto commit = []() { asm volatile("cp.async.commit_group;" ::: "memory"); };
    auto rows_of = [&](int e0) -> int4 {                               // rows of elements e0 .. e0+3
        return p.rmap ? __ldg(reinterpret_cast<const int4 *>(p.rmap + e0)) : make_int4(e0, e0 + 1, e0 + 2, e0 + 3);
    };
    // element (row, frame) of a step-major array sits at row * pitch + frame: 32-bit offsets (launch_map checks N * pitch)
    const uint32_t pitch32 = (uint32_t)p.pitch, f32 = (uint32_t)f;
    auto issue_group = [&](uint32_t dst, int e0, const int4 &r) {      // 12 floats -> dst + 4 bd k
        const int rr[G] = {r.x, r.y, r.z, r.w};
        const uint32_t op = (uint32_t)e0 * pitch32 + f32;
#pragma unroll
        for (int i = 0; i < G; ++i) {
            const uint32_t o = (uint32_t)rr[i] * pitch32 + f32;
            cp4(dst + 4u * bd * i, p.sys + o);
            cp4(dst + 4u * bd * (4 + i), p.par + (op + (uint32_t)i * pitch32));
            cp4(dst + 4u * bd * (8 + i), p.La + o);
        }
    };
    // a stream of `ng` groups, group n = elements first + n * stride .. +3, through the ring: start() fills the ring,
    // take(n) waits for group n, hands out its values and refills its slot with group n + RB
    int4 rnext = make_int4(0, 0, 0, 0);
    auto stream_start = [&](int first, int stride, int ng) {
#pragma unroll
        for (int k = 0; k < RB; ++k) {
            if (k < ng) issue_group(ring_s + 4u * bd * 12 * k, first + k * stride, rows_of(first + k * stride));
            commit();
        }
        if (RB < ng) rnext = rows_of(first + RB * stride);
    };
    auto stream_take = [&](int n, int slot, int first, int stride, int ng, float (&vs)[G], float (&vp)[G], float (&vl)[G]) {
        asm volatile("cp.async.wait_group %0;" ::"n"(RB - 1) : "memory");
        const float *q = ring + slot * 12 * bd + tid;
#pragma unroll
        for (int i = 0; i < G; ++i) { vs[i] = q[i * bd]; vp[i] = q[(4 + i) * bd]; vl[i] = q[(8 + i) * bd]; }
        // (the interleaver entries of the group after next are requested BEFORE this group's copies: behind twelve DRAM
        // misses in the load queue they came back too late -- 12 % of decoder 2's warp samples waited on them)
        const int4 rcur = rnext;
        if (n + RB + 1 < ng) rnext = rows_of(first + (n + RB + 1) * stride);
        if (n + RB < ng) issue_group(ring_s + 4u * bd * 12 * slot, first + (n + RB) * stride, rcur);
        commit();
    };
    // four beta steps (newest first: gw[3] is the latest step), rescaled at the end; the per-step form if they decayed
    auto beta_block = [&](float (&B)[S], const float4 (&gw)[G]) {
        float B0[S];
#pragma unroll
        for (int s = 0; s < S; ++s) B0[s] = B[s];
#pragma unroll
        for (int i = G - 1; i >= 0; --i) beta_raw(B, gw[i]);
        float sum = total(B);
        if (!(sum >= RESCALE_FLOOR)) {
#pragma unroll
            for (int s = 0; s < S; ++s) B[s] = B0[s];
#pragma unroll
            for (int i = G - 1; i >= 0; --i) { beta_raw(B, gw[i]); scale(B, total(B)); }
            sum = total(B);
        }
        scale(B, sum);
    };

    // ---- backward sweep with checkpoints (the metrics are scaled to sum 1 at every multiple of 4 steps)
    {
        float B[S];
        const int tb = min(N, hi + WARM);
#pragma unroll
        for (int s = 0; s < S; ++s) B[s] = 1.0f / S;                      // beta_N = 1 for all states (:225-226), scale free
        // The inputs of a group (4 steps) are fetched two groups ahead of their use into one of TWO statically named
        // register sets, the loop handles both per iteration.  (A rolled loop that rotates the sets by register moves makes
        // ptxas guard all of them with one scoreboard: the first use then waits for the loads issued half an iteration ago
        // -- 26 % of all warp samples sat on that instruction.)
        if constexpr (SM) {
            const int ng = (tb - lo) / G;
            stream_start(tb - G, -G, ng);
            int slot = 0;
#pragma unroll 1
            for (int n = 0; n < ng; ++n) {
                float vs[G], vp[G], vl[G];
                stream_take(n, slot, tb - G, -G, ng, vs, vp, vl);
                slot = (slot + 1 == RB) ? 0 : slot + 1;
                float4 gw[G];
#pragma unroll
                for (int i = 0; i < G; ++i) gw[i] = weights(vs[i], vp[i], vl[i]);
                const int e1 = tb - n * G;
                if (e1 <= hi && (((e1 - lo) % CK) == 0 || e1 == hi)) {        // beta_{e1}: the checkpoint of segment j
                    const int j = (e1 - lo + CK - 1) / CK - 1;
#pragma unroll
                    for (int s = 0; s < S; ++s) (ck + (uint32_t)(j * S) * NT32)[(uint32_t)s * NT32] = B[s];
                }
                beta_block(B, gw);
            }
        } else {
        float qs[2][G], qp[2][G], ql[2][G];
        ld3(tb - G, qs[0], qp[0], ql[0]);
        if (tb - G > lo) ld3(tb - 2 * G, qs[1], qp[1], ql[1]);
        auto group = [&](int e1, float (&vs)[G], float (&vp)[G], float (&vl)[G]) {
            float4 gw[G];
#pragma unroll
            for (int i = 0; i < G; ++i) gw[i] = weights(vs[i], vp[i], vl[i]);
            if (e1 - 2 * G > lo) ld3(e1 - 3 * G, vs, vp, vl);
            if (e1 <= hi && (((e1 - lo) % CK) == 0 || e1 == hi)) {        // beta_{e1}: the checkpoint of segment j
                const int j = (e1 - lo + CK - 1) / CK - 1;
#pragma unroll
                for (int s = 0; s < S; ++s) (ck + (uint32_t)(j * S) * NT32)[(uint32_t)s * NT32] = B[s];
            }
            beta_block(B, gw);
        };
#pragma unroll 1
        for (int e1 = tb; e1 > lo; e1 -= 2 * G) {
            group(e1, qs[0], qp[0], ql[0]);
            if (e1 - G > lo) group(e1 - G, qs[1], qp[1], ql[1]);
        }
        }
    }
    // ---- forward sweep
    float A[S];
    const int ta = max(0, lo - WARM);
#pragma unroll
    for (int s = 0; s < S; ++s) A[s] = (ta == 0) ? ((s == 0) ? 1.0f : 0.0f) : (1.0f / S);    // alpha_0 = delta(s,0), :220-221
    // one alpha step; with EMIT the a-posteriori log2 ratio of the step (prior included) from the beta words bt[0..SV)
    bool small = false;
    auto alpha_raw = [&](float (&A_)[S], const float4 &gw, const float4 *bt, bool emit, float &D, bool rescue = false) {
        float tx[2 * S];
#pragma unroll
        for (int e = 0; e < 2 * S; ++e) tx[e] = A_[e >> 1] * pick(gw, T::out(e >> 1, e & 1));
        if (emit) {
            float bv[S];
#pragma unroll
            for (int v = 0; v < SV; ++v) {
                const float4 q = bt[v * bd];
                bv[4 * v] = q.x; bv[4 * v + 1] = q.y; bv[4 * v + 2] = q.z; bv[4 * v + 3] = q.w;
            }
            float a0 = 0.0f, a1 = 0.0f, c0 = 0.0f, c1 = 0.0f;       // two partial sums each: shorter dependency chains
#pragma unroll
            for (int s = 0; s < S; s += 2) {
                a0 += tx[2 * s] * bv[T::ns(s, 0)];
                a1 += tx[2 * s + 1] * bv[T::ns(s, 1)];
                c0 += tx[2 * s + 2] * bv[T::ns(s + 1, 0)];
                c1 += tx[2 * s + 3] * bv[T::ns(s + 1, 1)];
            }
            a0 += c0; a1 += c1;
            // both sums below 2^-40 (contradicted observations): the block is redone with `rescue`, which takes the sums 2^80 up
            small = small || (fmaxf(a0, a1) < 9.094947017729282e-13f);
            if (rescue && fmaxf(a0, a1) < 9.094947017729282e-13f) {
                a0 = a1 = 0.0f;
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    a0 += (tx[2 * s] * 1.099511627776e12f) * (bv[T::ns(s, 0)] * 1.099511627776e12f);
                    a1 += (tx[2 * s + 1] * 1.099511627776e12f) * (bv[T::ns(s, 1)] * 1.099511627776e12f);
                }
            }
            D = lg2(fmaxf(a1, 1.0e-37f)) - lg2(fmaxf(a0, 1.0e-37f));
        }
#pragma unroll
        for (int n = 0; n < S; ++n) A_[n] = tx[T::pred(n, 0)] + tx[T::pred(n, 1)];             // :136-138
    };
    // step-major: the first segment's inputs and checkpoint are requested before the warm-up, segment j+1's when segment j
    // has been read out of `segbuf` (32 floats: 2 x 12 inputs, 8 checkpoint values)
    int4 rc[2], rn[2];                          // rows of the current / the next segment (the interleaver entries are
                                                // loaded a segment before the addresses they form are needed)
    rc[0] = rc[1] = rn[0] = rn[1] = make_int4(0, 0, 0, 0);
    auto segment_rows = [&](int s0, int4 (&r)[2]) {
        const int ns = min(CK, hi - s0);
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (h * G < ns) r[h] = rows_of(s0 + h * G);
    };
    auto issue_segment = [&](int s0, int j, const int4 (&r)[2]) {
        const int ns = min(CK, hi - s0);
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (h * G < ns) issue_group(seg_s + 4u * bd * 12 * h, s0 + h * G, r[h]);
#pragma unroll
        for (int s = 0; s < S; ++s) cp4(seg_s + 4u * bd * (24 + s), (ck + (uint32_t)(j * S) * NT32) + (uint32_t)s * NT32);
        commit();
    };
    if constexpr (SM) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");   // (only empty groups are pending: the ring's slots are free)
        if (lo < hi) { segment_rows(lo, rn); issue_segment(lo, 0, rn); }
        stream_start(ta, G, (lo - ta) / G);
    }
    int wslot = 0;
    for (int e0 = ta; e0 < lo; e0 += G) {                       // warm-up (no LLRs, no beta)
        float vs[G], vp[G], vl[G];
        if constexpr (SM) {
            stream_take((e0 - ta) / G, wslot, ta, G, (lo - ta) / G, vs, vp, vl);
            wslot = (wslot + 1 == RB) ? 0 : wslot + 1;
        } else {
            ld3(e0, vs, vp, vl);
        }
        float4 gw[G];
#pragma unroll
        for (int i = 0; i < G; ++i) gw[i] = weights(vs[i], vp[i], vl[i]);
        float A0[S], dummy;
#pragma unroll
        for (int s = 0; s < S; ++s) A0[s] = A[s];
#pragma unroll
        for (int i = 0; i < G; ++i) alpha_raw(A, gw[i], nullptr, false, dummy);
        float sum = total(A);
        if (!(sum >= RESCALE_FLOOR)) {
#pragma unroll
            for (int s = 0; s < S; ++s) A[s] = A0[s];
#pragma unroll
            for (int i = 0; i < G; ++i) { alpha_raw(A, gw[i], nullptr, false, dummy); scale(A, total(A)); }
            sum = total(A);
        }
        scale(A, sum);
    }
    // the inputs and the beta checkpoint of a segment are fetched while the previous segment is being processed
    static_assert(CK == 2 * G, "segment = two vector groups");
    float xin[2][3][G], xck[S];
    auto fetch_segment = [&](int s0, int j) {
        const int ns = min(CK, hi - s0);
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (h * G < ns) ld3(s0 + h * G, xin[h][0], xin[h][1], xin[h][2]);
#pragma unroll
        for (int s = 0; s < S; ++s) xck[s] = (ck + (uint32_t)(j * S) * NT32)[(uint32_t)s * NT32];
    };
    if constexpr (!SM) {
        if (lo < hi) fetch_segment(lo, 0);
    }
    for (int s0 = lo, j = 0; s0 < hi; s0 += CK, ++j) {
        const int ns = min(CK, hi - s0);                        // 4 or 8
        if constexpr (SM) {
            rc[0] = rn[0]; rc[1] = rn[1];
            if (s0 + CK < hi) segment_rows(s0 + CK, rn);
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            const float *q = segbuf + tid;
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int i = 0; i < G; ++i) xin[h][a][i] = q[(h * 12 + a * 4 + i) * bd];
#pragma unroll
            for (int s = 0; s < S; ++s) xck[s] = q[(24 + s) * bd];
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (h * G < ns) {
#pragma unroll
                for (int i = 0; i < G; ++i) {
                    sg[(h * G + i) * bd + tid] = weights(xin[h][0][i], xin[h][1][i], xin[h][2][i]);
                    sl[(h * G + i) * bd + tid] = xin[h][2][i];
                }
            }
        }
        float B[S];
#pragma unroll
        for (int s = 0; s < S; ++s) B[s] = xck[s];
        if constexpr (SM) {
            if (s0 + CK < hi) issue_segment(s0 + CK, j + 1, rn);
        } else {
            if (s0 + CK < hi) fetch_segment(s0 + CK, j + 1);
        }
        // beta of the segment, backwards from its checkpoint, block by block (beta_{s0+1+k} -> sb[k])
        auto store_beta = [&](int k, const float (&Bv)[S]) {
#pragma unroll
            for (int v = 0; v < SV; ++v) sb[(k * SV + v) * bd + tid] = make_float4(Bv[4 * v], Bv[4 * v + 1], Bv[4 * v + 2], Bv[4 * v + 3]);
        };
        for (int h = ns / G - 1; h >= 0; --h) {
            float B0[S];
#pragma unroll
            for (int s = 0; s < S; ++s) B0[s] = B[s];
            float4 gq[G];                                        // (read before the stores below, which the compiler must
#pragma unroll                                                   //  assume to alias them)
            for (int i = 0; i < G; ++i) gq[i] = sg[(h * G + i) * bd + tid];
#pragma unroll
            for (int i = G - 1; i >= 0; --i) { store_beta(h * G + i, B); beta_raw(B, gq[i]); }
            float sum = total(B);
            if (!(sum >= RESCALE_FLOOR)) {
#pragma unroll
                for (int s = 0; s < S; ++s) B[s] = B0[s];
#pragma unroll
                for (int i = G - 1; i >= 0; --i) {
                    store_beta(h * G + i, B); beta_raw(B, sg[(h * G + i) * bd + tid]); scale(B, total(B));
                }
                sum = total(B);
            }
            scale(B, sum);
        }
        // alpha / a-posteriori LLRs forwards, block by block
        for (int h = 0; h < ns / G; ++h) {
            float A0[S], Dv[G];
#pragma unroll
            for (int s = 0; s < S; ++s) A0[s] = A[s];
            small = false;
            float4 gq[G];
#pragma unroll
            for (int i = 0; i < G; ++i) gq[i] = sg[(h * G + i) * bd + tid];
#pragma unroll
            for (int i = 0; i < G; ++i) alpha_raw(A, gq[i], sb + (h * G + i) * SV * bd + tid, true, Dv[i]);
            float sum = total(A);
            if (!(sum >= RESCALE_FLOOR) || small) {
#pragma unroll
                for (int s = 0; s < S; ++s) A[s] = A0[s];
#pragma unroll
                for (int i = 0; i < G; ++i) {
                    alpha_raw(A, sg[(h * G + i) * bd + tid], sb + (h * G + i) * SV * bd + tid, true, Dv[i], true);
                    scale(A, total(A));
                }
                sum = total(A);
            }
            scale(A, sum);
            float Le[G], Lv[G];                                  // extrinsic L - L_int and the full LLR (:145)
#pragma unroll
            for (int i = 0; i < G; ++i) {
                const float la = sl[(h * G + i) * bd + tid];
                Le[i] = LN2 * (Dv[i] - fminf(fmaxf(la * LOG2E, -60.0f), 60.0f));
                Lv[i] = la + Le[i];
            }
            const int e0 = s0 + h * G;
            if (SM) {
                const int4 rr = (h == 0) ? rc[0] : rc[1];
                const int r[G] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
                for (int i = 0; i < G; ++i) {
                    const uint32_t o = (uint32_t)r[i] * pitch32 + f32;
                    p.L_out[o] = p.ext ? Le[i] : Lv[i];
                    if (p.bits_out) p.bits_out[o] = (uint8_t)(p.mode == 1 && Lv[i] > 0.0f);
                }
            } else {
                if (p.ext) *reinterpret_cast<float4 *>(p.L_out + f * N + e0) = make_float4(Le[0], Le[1], Le[2], Le[3]);
                else *reinterpret_cast<float4 *>(p.L_out + f * N + e0) = make_float4(Lv[0], Lv[1], Lv[2], Lv[3]);
                if (p.bits_out) {
                    uchar4 b;
                    b.x = (p.mode == 1 && Lv[0] > 0.0f); b.y = (p.mode == 1 && Lv[1] > 0.0f);
                    b.z = (p.mode == 1 && Lv[2] > 0.0f); b.w = (p.mode == 1 && Lv[3] > 0.0f);
                    *reinterpret_cast<uchar4 *>(p.bits_out + f * N + e0) = b;
                }
            }
        }
    }
}

// compile-time trellises the register-resident kernels are instantiated for (packed from commpy_b200's Trellis tables)
using RscK4 = CT<8, 0xedfc96369120ull, 0xc99cc99cu>;         // Trellis([3], [[1, 0o15]], [[0o13]], 'rsc')  (config C3)
using RscK4Legacy = CT<8, 0xedf5b2a4d120ull, 0xcc9999ccu>;   // Trellis([3], [[1, 0o15]], 0o13, 'rsc')
using RscK3Legacy = CT<4, 0x2d9090ull, 0x99ccu>;             // Trellis([2], [[1, 7]], 5, 'rsc')     (test_convcode.py:37)
using FfK3 = CT<4, 0x659410ull, 0x693cu>;                    // Trellis([2], [[5, 7]])
using RscK3 = CT<4, 0x64b090ull, 0x9c9cu>;                   // Trellis([2], [[1, 5]], [[7]], 'rsc')

template <class T>
static bool matches(const int32_t *next, const int32_t *out, int S)
{
    if (S != T::S) return false;
    for (int s = 0; s < S; ++s)
        for (int u = 0; u < 2; ++u)
            if (next[s * 2 + u] != T::ns(s, u) || out[s * 2 + u] != T::out(s, u)) return false;
    return true;
}

// calls fn(T()) with the compile-time trellis T whose tables are the host tables (next, out) and returns true; false when
// no compile-time trellis matches
template <class Fn>
static bool with_ct(const int32_t *next, const int32_t *out, int S, Fn &&fn)
{
    if (matches<RscK4>(next, out, S)) fn(RscK4());
    else if (matches<RscK4Legacy>(next, out, S)) fn(RscK4Legacy());
    else if (matches<RscK3Legacy>(next, out, S)) fn(RscK3Legacy());
    else if (matches<FfK3>(next, out, S)) fn(FfK3());
    else if (matches<RscK3>(next, out, S)) fn(RscK3());
    else return false;
    return true;
}

// steps per window: 1024 unless cpb_set_option(CPB_OPT_BCJR_WINDOW, w) asks for shorter windows (a multiple of 8, >= 128):
// more threads per frame for small batches at the price of more warm-up steps.  The split depends only on N and this
// explicit option, never on the batch, so a frame decodes identically whatever it is batched with.
static int window_len()
{
    int w = option(CPB_OPT_BCJR_WINDOW);
    if (w <= 0) return WIN;
    w = (w / 8) * 8;
    return std::min(4096, std::max(128, w));
}
static int nwindows(int N) { const int w = window_len(); return (N > w + w / 2) ? (int)ceil_div(N, w) : 1; }

// the checkpointed kernels read 16-byte vectors of a row (vec: N % 4 == 0 and aligned pointers) and work in blocks of 4
// steps (a window that is not a multiple of CK ends in a 4-step segment)
static bool blocked(bool vec, int win) { return vec && win % 4 == 0; }

// map_lin2_kernel is written for systematic trellises with 4 or 8 states ...
template <class T>
constexpr bool lin2_trellis = systematic<T>() && T::S % 4 == 0;

// ... and runs on them unless per-step scaling is asked for.  It is the only kernel that reads step-major arrays, so the
// turbo loop runs step-major exactly when it takes the trellis and the frame length (step_major_ok).
template <class T>
static bool lin2_ok(bool vec, int win)
{
    return lin2_trellis<T> && blocked(vec, win) && !option(CPB_OPT_BCJR_PER_STEP_SCALING);
}

template <class T>
static int launch(const Params &p, bool vec, cudaStream_t st)
{
    // the checkpointed kernels run one warp per CTA: 49,152 threads (C3: 8,192 frames x 6 windows) are 1,536 CTAs instead
    // of 384, which spreads evenly over 148 SMs (measured 0.88 vs 0.91 ms per pass)
    const int bd = 32;
    const unsigned grid = (unsigned)ceil_div(p.NT, bd);
    if constexpr (lin2_trellis<T>) {
        // (the kernel indexes its checkpoints with 32-bit offsets: always true for the chunks chunk_frames() makes)
        if (lin2_ok<T>(vec, p.win) && p.NT * (int64_t)(ceil_div(p.win, CK) * T::S) < (1ll << 31)) {
            // beta, weights and L_int of a segment; step-major: + the 32 staged floats of the next segment (the beta /
            // weight area doubles as the input ring of the backward sweep)
            const size_t smem2 = (size_t)bd * (CK * (T::S / 4 * sizeof(float4) + sizeof(float4) + sizeof(float)) +
                                               (p.pitch ? 32 * sizeof(float) : 0));
            void (*kern)(const Params) = p.pitch ? map_lin2_kernel<T, true> : map_lin2_kernel<T, false>;
            { const int rc_ = ensure_dyn_smem(reinterpret_cast<const void *>(kern), smem2, p.pitch != 0); if (rc_) return rc_; }
            kern<<<grid, bd, smem2, st>>>(p);
            CPB_LAUNCH_CHECK();
            return CPB_OK;
        }
    }
    if (p.pitch) return CPB_EINVAL;                  // step-major arrays: map_lin2_kernel only
    if (blocked(vec, p.win)) {
        const size_t smem = sizeof(float) * CK * (T::S + 3) * bd;
        { const int rc_ = ensure_dyn_smem(reinterpret_cast<const void *>(map_lin_kernel<T>), smem); if (rc_) return rc_; }
        map_lin_kernel<T><<<grid, bd, smem, st>>>(p);
    } else {
        map_tpf_kernel<T><<<(unsigned)ceil_div(p.NT, 128), 128, 0, st>>>(p);
    }
    CPB_LAUNCH_CHECK();
    return CPB_OK;
}

}  // namespace tpf

// out[f][i] = a[f][perm[i]] - (b ? b[f][perm[i]] : 0)        interleave (interleavers.py:13-29) of an extrinsic
__global__ void __launch_bounds__(256) gather_sub_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                         const int32_t *__restrict__ perm, int64_t batch, int N,
                                                         float *__restrict__ out)
{
    const int64_t total = batch * N;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t f = g / N;
        const int i = (int)(g - f * N);
        const int p = __ldg(&perm[i]);
        const float v = a[f * N + p] - (b ? b[f * N + p] : 0.0f);
        out[g] = v;
    }
}

// out[f][perm[i]] = a[f][i] - b[f][i]                          de-interleave (interleavers.py:31-47)
__global__ void __launch_bounds__(256) scatter_sub_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                          const int32_t *__restrict__ perm, int64_t batch, int N,
                                                          float *__restrict__ out)
{
    const int64_t total = batch * N;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t f = g / N;
        const int i = (int)(g - f * N);
        out[f * N + __ldg(&perm[i])] = a[g] - (b ? b[g] : 0.0f);
    }
}

// Row-staged forms of the three permutation kernels (one CTA per frame, the frame's row lives in shared memory):
// the global side is fully coalesced and the random access of the interleaver happens in shared memory.
// (The element-wise forms above issue one 32-byte sector request per 4-byte element: 0.35 ms per call at C3.)
__global__ void __launch_bounds__(256) row_gather_sub_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                             const int32_t *__restrict__ perm, int N, float *__restrict__ out)
{
    extern __shared__ float row[];
    const int64_t base = (int64_t)blockIdx.x * N;
    const bool v4 = ((N & 3) == 0) && ((((uintptr_t)(a + base)) | ((uintptr_t)(out + base)) | ((uintptr_t)perm) |
                                        (b ? (uintptr_t)(b + base) : 0)) & 15) == 0;
    if (v4) {                                                  // 16-byte global accesses, 4-byte shared-memory gathers
        const float4 *a4 = reinterpret_cast<const float4 *>(a + base);
        const float4 *b4 = b ? reinterpret_cast<const float4 *>(b + base) : nullptr;
        float4 *r4 = reinterpret_cast<float4 *>(row);
        for (int i = threadIdx.x; i < (N >> 2); i += blockDim.x) {
            float4 v = a4[i];
            if (b4) { const float4 w = b4[i]; v.x -= w.x; v.y -= w.y; v.z -= w.z; v.w -= w.w; }
            r4[i] = v;
        }
        __syncthreads();
        const int4 *p4 = reinterpret_cast<const int4 *>(perm);
        float4 *o4 = reinterpret_cast<float4 *>(out + base);
        for (int i = threadIdx.x; i < (N >> 2); i += blockDim.x) {
            const int4 q = __ldg(&p4[i]);
            o4[i] = make_float4(row[q.x], row[q.y], row[q.z], row[q.w]);
        }
        return;
    }
    for (int i = threadIdx.x; i < N; i += blockDim.x) row[i] = a[base + i] - (b ? b[base + i] : 0.0f);
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) out[base + i] = row[__ldg(&perm[i])];
}

__global__ void __launch_bounds__(256) row_scatter_sub_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                              const int32_t *__restrict__ perm, int N, float *__restrict__ out)
{
    extern __shared__ float row[];
    const int64_t base = (int64_t)blockIdx.x * N;
    const bool v4 = ((N & 3) == 0) && ((((uintptr_t)(a + base)) | ((uintptr_t)(out + base)) | ((uintptr_t)perm) |
                                        (b ? (uintptr_t)(b + base) : 0)) & 15) == 0;
    if (v4) {
        const float4 *a4 = reinterpret_cast<const float4 *>(a + base);
        const float4 *b4 = b ? reinterpret_cast<const float4 *>(b + base) : nullptr;
        const int4 *p4 = reinterpret_cast<const int4 *>(perm);
        for (int i = threadIdx.x; i < (N >> 2); i += blockDim.x) {
            float4 v = a4[i];
            if (b4) { const float4 w = b4[i]; v.x -= w.x; v.y -= w.y; v.z -= w.z; v.w -= w.w; }
            const int4 q = __ldg(&p4[i]);
            row[q.x] = v.x; row[q.y] = v.y; row[q.z] = v.z; row[q.w] = v.w;
        }
        __syncthreads();
        const float4 *r4 = reinterpret_cast<const float4 *>(row);
        float4 *o4 = reinterpret_cast<float4 *>(out + base);
        for (int i = threadIdx.x; i < (N >> 2); i += blockDim.x) o4[i] = r4[i];
        return;
    }
    for (int i = threadIdx.x; i < N; i += blockDim.x) row[__ldg(&perm[i])] = a[base + i] - (b ? b[base + i] : 0.0f);
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) out[base + i] = row[i];
}

__global__ void __launch_bounds__(256) row_scatter_bits_kernel(const uint8_t *__restrict__ a, const int32_t *__restrict__ perm,
                                                               int N, uint8_t *__restrict__ out)
{
    extern __shared__ uint8_t brow[];
    const int64_t base = (int64_t)blockIdx.x * N;
    for (int i = threadIdx.x; i < N; i += blockDim.x) brow[__ldg(&perm[i])] = a[base + i];
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) out[base + i] = brow[i];
}

__global__ void __launch_bounds__(256) scatter_bits_kernel(const uint8_t *__restrict__ a, const int32_t *__restrict__ perm,
                                                           int64_t batch, int N, uint8_t *__restrict__ out)
{
    const int64_t total = batch * N;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t f = g / N;
        const int i = (int)(g - f * N);
        out[f * N + __ldg(&perm[i])] = a[g];
    }
}

// (batch, N) frame-major floats -> (N, pitch) step-major: the layout the turbo loop works in (every access of the MAP
// kernel is then a full 128-byte line per warp and the interleaver is a row index, not a data movement)
__global__ void __launch_bounds__(256) to_step_major_kernel(const float *__restrict__ in, int64_t batch, int N, int64_t pitch,
                                                            float *__restrict__ out)
{
    __shared__ float tile[32][33];
    const int64_t f0 = (int64_t)blockIdx.y * 32;
    const int t0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int64_t f = f0 + r;
        const int t = t0 + tx;
        tile[r][tx] = (f < batch && t < N) ? in[f * N + t] : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int t = t0 + r;
        const int64_t f = f0 + tx;
        if (t < N && f < pitch) out[(int64_t)t * pitch + f] = tile[tx][r];
    }
}

// (N, pitch) step-major bytes -> (batch, N) frame-major (the decisions of the last MAP pass)
__global__ void __launch_bounds__(256) bits_to_frame_major_kernel(const uint8_t *__restrict__ in, int64_t batch, int N,
                                                                  int64_t pitch, uint8_t *__restrict__ out)
{
    __shared__ uint8_t tile[128][36];
    const int64_t f0 = (int64_t)blockIdx.y * 32;
    const int t0 = blockIdx.x * 128;
    for (int r = threadIdx.x >> 3; r < 128; r += 32) {           // 8 threads read the 32 bytes of a row
        const int q = threadIdx.x & 7;
        const int t = t0 + r;
        uint32_t w = 0u;
        if (t < N) w = *reinterpret_cast<const uint32_t *>(in + (int64_t)t * pitch + f0 + 4 * q);
        *reinterpret_cast<uint32_t *>(&tile[r][4 * q]) = w;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 32 * 128; i += 256) {
        const int fl = i >> 7, tl = i & 127;
        const int64_t f = f0 + fl;
        const int t = t0 + tl;
        if (f < batch && t < N) out[f * N + t] = tile[tl][fl];
    }
}

// floats of beta scratch one chunk of `frames` frames needs (whichever kernel runs)
static size_t beta_floats(int64_t frames, int N, int S)
{
    const int nwin = tpf::nwindows(N);
    const int win = (nwin == 1) ? N : tpf::window_len();
    const int64_t bp = ceil_div(frames, 32) * 32;
    const size_t a = (size_t)frames * (N + 1) * S;
    const size_t b = (size_t)nwin * bp * win * S;
    return std::max(a, b);
}

static int launch_map(const cpbTrellis *t, int S, const float *sys, const float *par, const float *La, int64_t batch,
                      int N, float noise_var, int mode, float *beta, float *L_out, uint8_t *bits, cudaStream_t st,
                      int want_ext = 0, int *did_ext = nullptr, int64_t pitch = 0, const int32_t *rmap = nullptr)
{
    const int32_t *hn = nullptr, *ho = nullptr;
    cpb_trellis_host_tables(t, &hn, &ho);
    tpf::Params p{};
    p.sys = sys; p.par = par; p.La = La; p.batch = batch; p.bp = ceil_div(batch, 32) * 32;
    p.N = N; p.nwin = tpf::nwindows(N); p.win = (p.nwin == 1) ? N : tpf::window_len();
    p.c = tpf::LOG2E / noise_var; p.mode = mode; p.beta = beta; p.NT = (int64_t)p.nwin * p.bp;
    p.L_out = L_out; p.bits_out = bits;
    const bool vec = (N % 4 == 0) && ((((uintptr_t)sys | (uintptr_t)par | (uintptr_t)La | (uintptr_t)L_out) & 15) == 0) &&
                     (bits == nullptr || (((uintptr_t)bits) & 3) == 0);
    p.ext = (want_ext && tpf::blocked(vec, p.win)) ? 1 : 0;
    p.pitch = pitch; p.rmap = rmap;
    if (pitch && (int64_t)N * pitch >= (1ll << 31)) return CPB_EINVAL;              // 32-bit element offsets in the kernel
    int rc = CPB_OK;
    if (tpf::with_ct(hn, ho, S, [&](auto ct) { rc = tpf::launch<decltype(ct)>(p, vec, st); })) {
        if (did_ext) *did_ext = p.ext;
        return rc;
    }
    if (pitch) return CPB_EINVAL;                    // step-major arrays: map_lin2_kernel only
    // any other rate-1/2 trellis with 2..32 states: table-driven lane-per-state kernel
    if (did_ext) *did_ext = 0;
    const int32_t *nx = cpb_trellis_next_dev(t), *ot = cpb_trellis_out_dev(t), *pd = cpb_trellis_pred_dev(t);
    const float inv2s2 = 1.0f / (2.0f * noise_var);
    const int fpw = 32 / S;
    const int64_t warps = ceil_div(batch, fpw);
    const unsigned grid = (unsigned)ceil_div(warps, 4);
#define CPB_MAP(SS) case SS: map_kernel<SS><<<grid, 128, 0, st>>>(sys, par, La, batch, N, nx, ot, pd, inv2s2, mode, beta, L_out, bits); break;
    switch (S) {
        CPB_MAP(2) CPB_MAP(4) CPB_MAP(8) CPB_MAP(16) CPB_MAP(32)
    default: return CPB_EUNSUPPORTED;
    }
#undef CPB_MAP
    CPB_LAUNCH_CHECK();
    return CPB_OK;
}

static int check_trellis(const cpbTrellis *t, int *S)
{
    if (!t) return CPB_EINVAL;
    int k, n;
    cpb_trellis_dims(t, &k, &n, S);
    if (k != 1 || n != 2) return CPB_EINVAL;              // map_decode is written for rate-1/2 codes (turbo.py:165-166)
    if (*S != 2 && *S != 4 && *S != 8 && *S != 16 && *S != 32) return CPB_EUNSUPPORTED;
    return CPB_OK;
}

// the turbo loop runs on step-major arrays when the block-rescaled kernel takes the trellis and the frame length (the
// arrays are the 16-byte aligned workspace; the kernel reads the interleaver as int4)
static bool step_major_ok(const cpbTrellis *t, int S, int N, const int32_t *perm_dev)
{
    if (option(CPB_OPT_TURBO_FRAME_MAJOR)) return false;
    const bool vec = (N % 4 == 0) && (reinterpret_cast<uintptr_t>(perm_dev) & 15) == 0;
    const int win = (tpf::nwindows(N) == 1) ? N : tpf::window_len();
    const int32_t *hn = nullptr, *ho = nullptr;
    cpb_trellis_host_tables(t, &hn, &ho);
    bool ok = false;
    tpf::with_ct(hn, ho, S, [&](auto ct) { ok = tpf::lin2_ok<decltype(ct)>(vec, win); });
    return ok;
}

static int64_t chunk_frames(int64_t batch, int N, int S)
{
    const double per = (double)(N + tpf::WIN + 1) * S * 4.0 + 5.0 * N * 4.0 + N;
    int64_t c = (int64_t)(6.0e9 / per);
    if (c < 1) c = 1;
    return std::min<int64_t>(c, batch);
}

}  // namespace bcjr

extern "C" {

int cpb_map_workspace_bytes(const cpbTrellis *t, int64_t batch, int64_t N, size_t *bytes)
{
    int S = 0;
    int rc = bcjr::check_trellis(t, &S);
    if (rc) return rc;
    if (!bytes || batch < 0 || N < 1 || N > (1 << 24)) return CPB_EINVAL;
    *bytes = batch ? bcjr::beta_floats(bcjr::chunk_frames(batch, (int)N, S), (int)N, S) * sizeof(float) : 0;
    return CPB_OK;
}

int cpb_turbo_workspace_bytes(const cpbTrellis *t, int64_t batch, int64_t N, size_t *bytes)
{
    int S = 0;
    int rc = bcjr::check_trellis(t, &S);
    if (rc) return rc;
    if (!bytes || batch < 0 || N < 1 || N > (1 << 24)) return CPB_EINVAL;
    const int64_t Fc = batch ? bcjr::chunk_frames(batch, (int)N, S) : 0;
    const size_t nvec = (size_t)ceil_div(Fc, 32) * 32 * N;     // the step-major arrays are padded to 32 frames
    *bytes = batch ? (bcjr::beta_floats(Fc, (int)N, S) + 5 * nvec) * sizeof(float) + nvec + 256 : 0;
    return CPB_OK;
}

int cpb_map_decode(const cpbTrellis *t, const float *sys_dev, const float *par_dev, const float *L_int_dev,
                   int64_t batch, int64_t N, float noise_variance, int mode, float *L_out_dev, uint8_t *bits_out_dev,
                   void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int S = 0;
    int rc = bcjr::check_trellis(t, &S);
    if (rc) return rc;
    if (batch == 0) return CPB_OK;
    if (!sys_dev || !par_dev || !L_int_dev || !L_out_dev || batch < 0 || N < 1 || N > (1 << 24) || !(noise_variance > 0.0f))
        return CPB_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t Fc = bcjr::chunk_frames(batch, (int)N, S);
    Scratch ws;
    rc = ws.acquire(workspace_dev, workspace_bytes, bcjr::beta_floats(Fc, (int)N, S) * sizeof(float), st);
    if (rc) return rc;
    for (int64_t f0 = 0; f0 < batch && rc == CPB_OK; f0 += Fc) {
        const int64_t nb = std::min<int64_t>(Fc, batch - f0);
        rc = bcjr::launch_map(t, S, sys_dev + f0 * N, par_dev + f0 * N, L_int_dev + f0 * N, nb, (int)N, noise_variance,
                              mode, reinterpret_cast<float *>(ws.ptr), L_out_dev + f0 * N,
                              bits_out_dev ? bits_out_dev + f0 * N : nullptr, st);
    }
    ws.release();
    return rc;
}

int cpb_turbo_decode(const cpbTrellis *t, const float *sys_dev, const float *par1_dev, const float *par2_dev,
                     const int32_t *perm_dev, int64_t batch, int64_t N, float noise_variance, int n_iter,
                     const float *L_int0_dev, uint8_t *bits_out_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int S = 0;
    int rc = bcjr::check_trellis(t, &S);
    if (rc) return rc;
    if (!sys_dev || !par1_dev || !par2_dev || !perm_dev || !bits_out_dev || batch < 0 || N < 1 || N > (1 << 24) ||
        n_iter < 0 || !(noise_variance > 0.0f))
        return CPB_EINVAL;
    if (batch == 0) return CPB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const DeviceProps &dp = device_props();
    const int64_t Fc = bcjr::chunk_frames(batch, (int)N, S);
    const size_t nbeta = bcjr::beta_floats(Fc, (int)N, S), nvec = (size_t)ceil_div(Fc, 32) * 32 * N;
    const bool step_major = bcjr::step_major_ok(t, S, (int)N, perm_dev);
    Scratch ws;
    rc = ws.acquire(workspace_dev, workspace_bytes, (nbeta + 5 * nvec) * sizeof(float) + nvec + 256, st);
    if (rc) return rc;
    float *beta = reinterpret_cast<float *>(ws.ptr);
    float *sys_i = beta + nbeta, *La1 = sys_i + nvec, *La2 = La1 + nvec, *L1 = La2 + nvec, *L2 = L1 + nvec;
    uint8_t *dec = reinterpret_cast<uint8_t *>(L2 + nvec);
    for (int64_t f0 = 0; f0 < batch && rc == CPB_OK; f0 += Fc) {
        const int64_t nb = std::min<int64_t>(Fc, batch - f0);
        const int64_t tot = nb * N;
        const unsigned eg = (unsigned)std::min<int64_t>(ceil_div(tot, 256), (int64_t)dp.sm_count * 32);
        const float *sy = sys_dev + f0 * N, *p1 = par1_dev + f0 * N, *p2 = par2_dev + f0 * N;
        cudaError_t e;
        if (step_major) {
            // sys_i = sysT, La1 / La2 = the two extrinsic arrays, L1 / L2 = parity 1 / 2, all (N, pitch); decT = `dec`
            const int64_t pitch = ceil_div(nb, 32) * 32;
            float *sysT = sys_i, *p1T = L1, *p2T = L2;
            const dim3 tg((unsigned)ceil_div(N, 32), (unsigned)(pitch / 32));
            bcjr::to_step_major_kernel<<<tg, 256, 0, st>>>(sy, nb, (int)N, pitch, sysT);
            bcjr::to_step_major_kernel<<<tg, 256, 0, st>>>(p1, nb, (int)N, pitch, p1T);
            bcjr::to_step_major_kernel<<<tg, 256, 0, st>>>(p2, nb, (int)N, pitch, p2T);
            if (L_int0_dev) { bcjr::to_step_major_kernel<<<tg, 256, 0, st>>>(L_int0_dev + f0 * N, nb, (int)N, pitch, La1); e = cudaGetLastError(); }
            else e = cudaMemsetAsync(La1, 0, (size_t)N * pitch * sizeof(float), st);                  // turbo.py:304-307
            if (e == cudaSuccess) e = cudaMemsetAsync(dec, 0, (size_t)N * pitch, st);
            if (e != cudaSuccess) { rc = record_cuda_error(e, "turbo init", __FILE__, __LINE__); break; }
            for (int it = 0; it < n_iter && rc == CPB_OK; ++it) {
                // decoder 1 in natural order (:315); decoder 2 reads the systematic stream and decoder 1's extrinsic through
                // the interleaver (:310,:318-319) and writes its own extrinsic / decisions back through it (:328-331)
                rc = bcjr::launch_map(t, S, sysT, p1T, La1, nb, (int)N, noise_variance, 0, beta, La2, nullptr, st, 1, nullptr,
                                      pitch, nullptr);
                if (rc) break;
                const int mode = (it == n_iter - 1) ? 1 : 0;                                            // :320-323
                rc = bcjr::launch_map(t, S, sysT, p2T, La2, nb, (int)N, noise_variance, mode, beta, La1, dec, st, 1, nullptr,
                                      pitch, perm_dev);
            }
            if (rc) break;
            const dim3 bg((unsigned)ceil_div(N, 128), (unsigned)(pitch / 32));
            bcjr::bits_to_frame_major_kernel<<<bg, 256, 0, st>>>(dec, nb, (int)N, pitch, bits_out_dev + f0 * N);
            e = cudaGetLastError();
            if (e != cudaSuccess) rc = record_cuda_error(e, "turbo kernels", __FILE__, __LINE__);
            continue;
        }
        if (L_int0_dev) e = cudaMemcpyAsync(La1, L_int0_dev + f0 * N, tot * sizeof(float), cudaMemcpyDeviceToDevice, st);
        else e = cudaMemsetAsync(La1, 0, tot * sizeof(float), st);                         // turbo.py:304-307
        if (e == cudaSuccess) e = cudaMemsetAsync(dec, 0, tot, st);
        if (e != cudaSuccess) { rc = record_cuda_error(e, "turbo init", __FILE__, __LINE__); break; }
        const bool rows = (size_t)N * sizeof(float) <= 96 * 1024;
        const size_t rsm = (size_t)N * sizeof(float);
        if (rows) {
            rc = ensure_dyn_smem(reinterpret_cast<const void *>(bcjr::row_gather_sub_kernel), rsm);
            if (!rc) rc = ensure_dyn_smem(reinterpret_cast<const void *>(bcjr::row_scatter_sub_kernel), rsm);
            if (!rc) rc = ensure_dyn_smem(reinterpret_cast<const void *>(bcjr::row_scatter_bits_kernel), (size_t)N);
            if (rc) break;
        }
        if (rows) bcjr::row_gather_sub_kernel<<<(unsigned)nb, 256, rsm, st>>>(sy, nullptr, perm_dev, (int)N, sys_i);
        else bcjr::gather_sub_kernel<<<eg, 256, 0, st>>>(sy, nullptr, perm_dev, nb, (int)N, sys_i);          // :310
        for (int it = 0; it < n_iter && rc == CPB_OK; ++it) {
            // when the probability-domain kernel runs it writes L - L_int itself (did = 1) and the permutation kernels
            // read one array instead of two
            int did = 0;
            rc = bcjr::launch_map(t, S, sy, p1, La1, nb, (int)N, noise_variance, 0, beta, L1, nullptr, st, 1, &did);   // :315
            if (rc) break;
            if (rows) bcjr::row_gather_sub_kernel<<<(unsigned)nb, 256, rsm, st>>>(L1, did ? nullptr : La1, perm_dev, (int)N, La2);
            else bcjr::gather_sub_kernel<<<eg, 256, 0, st>>>(L1, did ? nullptr : La1, perm_dev, nb, (int)N, La2);   // :318-319
            const int mode = (it == n_iter - 1) ? 1 : 0;                                                // :320-323
            rc = bcjr::launch_map(t, S, sys_i, p2, La2, nb, (int)N, noise_variance, mode, beta, L2, dec, st, 1, &did);  // :326
            if (rc) break;
            if (rows) bcjr::row_scatter_sub_kernel<<<(unsigned)nb, 256, rsm, st>>>(L2, did ? nullptr : La2, perm_dev, (int)N, La1);
            else bcjr::scatter_sub_kernel<<<eg, 256, 0, st>>>(L2, did ? nullptr : La2, perm_dev, nb, (int)N, La1);   // :328-329
        }
        if (rc) break;
        if (rows) bcjr::row_scatter_bits_kernel<<<(unsigned)nb, 256, (size_t)N, st>>>(dec, perm_dev, (int)N, bits_out_dev + f0 * N);
        else bcjr::scatter_bits_kernel<<<eg, 256, 0, st>>>(dec, perm_dev, nb, (int)N, bits_out_dev + f0 * N); // :331
        e = cudaGetLastError();
        if (e != cudaSuccess) rc = record_cuda_error(e, "turbo kernels", __FILE__, __LINE__);
    }
    ws.release();
    return rc;
}

}  // extern "C"
