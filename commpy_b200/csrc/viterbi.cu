// Viterbi decoding on sm_100a -- replaces the loop nest of commpy/channelcoding/convcode.py:661-749
// (viterbi_decode), :590-657 (_acs_traceback), :575-587 (_compute_branch_metrics), :561-572 (_where_c).
//
// Exact semantics kept from the reference (SURVEY.md App. A.1):
//   * T = int((L+M)/k) - 1 trellis steps, zero / -1 padding past the received data;
//   * add-compare-select picks the FIRST minimum in (prev_state asc, input asc) order;
//   * the symbol of step q is read on the survivor path that starts at the lowest-index best state of
//     step min(q + D - 2, T) (D = tb_depth): one sliding-window traceback per output symbol.
//
// Two kernel families:
//   viterbi_fast_kernel     k=1, n=2 feed-forward shift-register codes with 64 states (K=7): one thread owns
//                           all 64 path metrics of one frame (int32 fixed-point LLR metrics) or of TWO frames
//                           (hard decision, u16x2-packed).  A key is metric << 10 | path history, so ONE add and ONE
//                           VIADDMNMX per state and step do add + compare + select with the reference tie rule AND
//                           record the survivor (register exchange over blocks of 4 steps); the best state of a
//                           step is a VIMNMX3 tree over the same keys.  Every 4 steps a 4-bit jump pointer per state
//                           goes to a shared-memory ring; the traceback jumps 4 steps per look-up.
//   viterbi_generic_kernel  any trellis (k<=4, n<=4, S<=256): table driven, one thread per frame, fp32 metrics
//                           in shared memory, survivors in a global scratch buffer.
// Both trace back in blocks of windows: one shared walk per block plus a fallback walk for every window whose own
// best state is not on it, which reproduces the reference's per-step traceback bit for bit.
#include <algorithm>
#include <cstdlib>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "handles.cuh"

using namespace cpb;


// ------------------------------------------------------------------------------------------------
// compile-time description of a rate-1/2 feed-forward code in CommPy's Trellis convention
// (convcode.py:195-255, polynomial_format='MSB'): generator bit b multiplies delay b (bit 0 = current
// input); state bit (M-b) holds delay b; output symbol = (parity(G0)<<1) | parity(G1).
// ------------------------------------------------------------------------------------------------
template <int M_, uint32_t G0_, uint32_t G1_>
struct FFCode {
    static constexpr int M = M_;
    static constexpr int S = 1 << M_;
    static constexpr uint32_t G0 = G0_, G1 = G1_;
    __host__ __device__ static constexpr int parity(uint32_t v)
    {
        v ^= v >> 16; v ^= v >> 8; v ^= v >> 4; v ^= v >> 2; v ^= v >> 1;
        return (int)(v & 1u);
    }
    __host__ __device__ static constexpr uint32_t regs(int s, int u)
    {
        uint32_t v = (uint32_t)u;
        for (int b = 1; b <= M_; ++b) v |= (uint32_t)((s >> (M_ - b)) & 1) << b;
        return v;
    }
    __host__ __device__ static constexpr int out(int s, int u)
    {
        return (parity(regs(s, u) & G0_) << 1) | parity(regs(s, u) & G1_);
    }
};

using Code133_171 = FFCode<6, 0133, 0171>;   // the standard K=7 code (octal 133,171)
using Code171_133 = FFCode<6, 0171, 0133>;
using Code5_43 = FFCode<6, 5, 43>;           // what Trellis makes of DECIMAL (133,171): wifi80211.py:49 quirk
using Code5_7 = FFCode<6, 5, 7>;             // the 64-state trellis of commpy/channelcoding/README.md:81-84 ([[5, 7]], memory 6)

template <class CODE>
static bool code_matches(const cpbTrellis &t)
{
    if (t.k != 1 || t.n != 2 || t.M != CODE::M || t.S != CODE::S) return false;
    for (int s = 0; s < CODE::S; ++s)
        for (int u = 0; u < 2; ++u) {
            if (t.next_state[s * 2 + u] != ((u << (CODE::M - 1)) | (s >> 1))) return false;
            if (t.output[s * 2 + u] != CODE::out(s, u)) return false;
        }
    return true;
}

// ------------------------------------------------------------------------------------------------
// Fast path: history-key add-compare-select + jump traceback (tests/model_jump_viterbi.py is the NumPy model)
//
//   key    = metric << FB | field                      FB = 6 + B history bits, B = 4 trellis steps per block
//   field  bit i <-> input u_{t0-5+i} on the state's survivor path (t0 = last block boundary): bits 0..5 are the
//          survivor's state at t0, bit 6+j is the input of sub-step j of the running block
//   ACS    Kn[l + 32u] = min(K[2l] + Bm[out(2l,u)], K[2l+1] + Bm[out(2l+1,u)]) + (u << (6+j))
//          ONE add and ONE add-min (VIADDMNMX) per state and step.  The smaller key wins; on equal metrics the
//          fields decide: both candidates carry the same newer history bits and differ in the predecessor's LSB,
//          so predecessor 2l wins -- the reference's first minimum over (prev_state asc) (convcode.py:612-642).
//   best   the minimum of the 64 keys: lowest metric, ties -> lowest field = lowest state index (np.argmin, :645);
//          its field is the best state's whole path back to the block boundary.
//   block  every B steps the low B bits of each key (the survivor's inputs u_{t0-5}..u_{t0-2}: a B-step jump
//          pointer) go to the shared-memory ring and the key becomes metric | state.
//   traceback  bit p is read on the path from best[min(p+D-1, T)] (App. A.1-8): start from that best key's
//          field, then jump B steps per look-up: state(t0-B) = ((state(t0) & 3) << 4) | nibble[t0][state(t0)].
// ------------------------------------------------------------------------------------------------
namespace fast {

constexpr int B = 4;               // trellis steps per history block
constexpr int FB = 6 + B;          // history bits in a key
constexpr int BD = 32;             // one warp per CTA: every synchronisation below is a __syncwarp()
constexpr int QBITS = 17;          // soft / unquantized: |quantised value| <= 2^17 (22 metric bits: 27 * 2^17 < 2^22)
constexpr int QMAX = 1 << QBITS;
constexpr int DMAX = 46;           // deepest traceback the fast path takes
constexpr int TASK_CAP = 384;      // retired paths kept per block and warp; beyond that they are finished inline
constexpr int TBB = 24;            // windows per traceback block (multiple of B, <= 28), hard and soft kernels alike
static_assert(TBB % 8 == 0, "bit-packed output: whole output bytes per traceback block");

struct Params {
    const void *coded;
    int64_t n_in;
    int64_t batch;
    int L, T, D;
    int TBB, NJ, RB;             // windows per traceback block, jumps below a block, ring blocks
    int mode;                    // CPB_VITERBI_*
    const float *frame_scale;    // float input: power-of-two scale per frame (device)
    uint8_t *out;
    int out_vec8;                // 1: rows of out are 8-byte aligned; 2: out is bit-packed (np.packbits order), L/8 bytes per row
    int in_aligned;              // 1: rows of coded are 4-byte (u8) / 16-byte (f32) aligned
    uint32_t met_mask;           // metric bits of a key, passed at run time so the key refresh stays one LOP3
    // punctured float input (IOP = 2): row of n_kept values; coded position c holds the next kept value when bit
    // (c mod punct_len) of punct_mask is set, else the erasure 0.0 (convcode.py:777-804)
    uint32_t punct_mask;
    int punct_len;
    int64_t n_kept;
};

template <int PACK> struct KeyOps;
template <> struct KeyOps<2> {   // two frames per register, u16 halves: 6 metric bits + 10 history bits
    static constexpr uint32_t FMASK = 0x03FF03FFu;
    static constexpr uint32_t INC0 = 0x00400040u;      // history bit 6 of both halves
    static constexpr uint32_t NIBM = 0x000F000Fu;
    __device__ static __forceinline__ uint32_t addmin(uint32_t a, uint32_t b, uint32_t c) { return __viaddmin_u16x2(a, b, c); }
    __device__ static __forceinline__ uint32_t min3(uint32_t a, uint32_t b, uint32_t c) { return __vimin3_u16x2(a, b, c); }
    __device__ static __forceinline__ uint32_t min2(uint32_t a, uint32_t b) { return __vminu2(a, b); }
    __device__ static __forceinline__ uint32_t idx(int s) { return (uint32_t)s | ((uint32_t)s << 16); }
};
template <> struct KeyOps<1> {   // one frame per register: 22 metric bits + 10 history bits
    static constexpr uint32_t FMASK = 0x3FFu;
    static constexpr uint32_t INC0 = 0x40u;
    static constexpr uint32_t NIBM = 0xFu;
    __device__ static __forceinline__ uint32_t addmin(uint32_t a, uint32_t b, uint32_t c) { return __viaddmin_u32(a, b, c); }
    __device__ static __forceinline__ uint32_t min3(uint32_t a, uint32_t b, uint32_t c) { return __vimin3_u32(a, b, c); }
    __device__ static __forceinline__ uint32_t min2(uint32_t a, uint32_t b) { return min(a, b); }
    __device__ static __forceinline__ uint32_t idx(int s) { return (uint32_t)s; }
};

// one trellis step on register-resident keys: Kn <- ACS(K, Bm); returns the minimum key(s)
template <class CODE, int PACK>
__device__ __forceinline__ uint32_t acs_step(const uint32_t (&K)[64], uint32_t (&Kn)[64], const uint32_t (&Bm)[4],
                                             const uint32_t inc)
{
    using OPS = KeyOps<PACK>;
    constexpr int H = CODE::S / 2;
    uint32_t Bm1[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) Bm1[o] = Bm[o] + inc;       // input 1 enters the history of the states l + H
#pragma unroll
    for (int l = 0; l < H; ++l) {
        const uint32_t c0 = K[2 * l + 1] + Bm[CODE::out(2 * l + 1, 0)];
        Kn[l] = OPS::addmin(K[2 * l], Bm[CODE::out(2 * l, 0)], c0);
        const uint32_t c1 = K[2 * l + 1] + Bm1[CODE::out(2 * l + 1, 1)];
        Kn[l + H] = OPS::addmin(K[2 * l], Bm1[CODE::out(2 * l, 1)], c1);
    }
    uint32_t r[22];
#pragma unroll
    for (int i = 0; i < 21; ++i) r[i] = OPS::min3(Kn[3 * i], Kn[3 * i + 1], Kn[3 * i + 2]);
    r[21] = Kn[63];
    uint32_t q[8];
#pragma unroll
    for (int i = 0; i < 7; ++i) q[i] = OPS::min3(r[3 * i], r[3 * i + 1], r[3 * i + 2]);
    q[7] = r[21];
    const uint32_t a = OPS::min3(q[0], q[1], q[2]);
    const uint32_t b = OPS::min3(q[3], q[4], q[5]);
    return OPS::min3(a, b, OPS::min2(q[6], q[7]));
}

// shared memory of one warp-CTA (byte offsets into smem_raw, so every access below compiles to LDS / STS / ATOMS)
extern __shared__ __align__(16) unsigned char smem_raw[];
template <int PACK>
struct Smem {
    static constexpr int NW = 8 * PACK;     // 32-bit words of jump nibbles per block and thread
    int nib;        // jump nibbles [RB][NW][32] u32: word w = states 4w..4w+3 (frame A low half, B high half) when
                    // PACK = 2, states 8w..8w+7 when PACK = 1
    int bf;         // best fields of the running traceback block [TBB/4][32] uint4 (one component per sub-step,
                    // frame B in the high half)
    int lut;        // hard-decision branch metrics [16] uint4
    int tasks;      // retired-path tasks [TASK_CAP] uint2
    int outbits;    // [32*PACK] u32
    int RB;
};
template <typename T> __device__ __forceinline__ T &sm_at(int off) { return *reinterpret_cast<T *>(smem_raw + off); }

static size_t smem_bytes(int RB, int TBB, int pack)
{
    size_t b = (size_t)RB * 8 * pack * BD * sizeof(uint32_t);
    b += (size_t)TBB * BD * sizeof(uint32_t);
    b += 16 * sizeof(uint4);
    b += (size_t)2 * (TASK_CAP + BD) * sizeof(uint32_t);       // + one scratch slot per lane
    b += (size_t)BD * pack * sizeof(uint32_t);
    return b;
}

// A survivor path as a shift register: bit i of `reg` is the input u_{t0-5+i}; one look-up moves t0 down by B steps.
template <int PACK, typename PT>
struct Jumper {
    static constexpr int ROWB = 8 * PACK * BD * 4;      // bytes per ring block
    int base, rowoff, wrap, fish;                       // base = ring offset + 4 * column
    PT reg;
    __device__ __forceinline__ void init(const Smem<PACK> &sm, int slot, int col, int fi, PT r0)
    {
        base = sm.nib + col * 4; rowoff = slot * ROWB; wrap = sm.RB * ROWB; fish = 16 * fi; reg = r0;
    }
    __device__ __forceinline__ void jump()
    {
        const uint32_t st = (uint32_t)reg & 63u;
        const int wsel = (PACK == 2) ? (int)((st >> 2) << 7) : (int)((st >> 3) << 7);
        const uint32_t sh = (PACK == 2) ? (((st & 3u) << 2) | (uint32_t)fish) : ((st & 7u) << 2);
        const uint32_t word = sm_at<uint32_t>(base + rowoff + wsel);
        reg = (PT)(reg << B) | (PT)((word >> sh) & 15u);
        rowoff -= ROWB;
        if (rowoff < 0) rowoff += wrap;
    }
};

// block bits of a path: it served the windows (lo, hi] and was retired in the block above boundary ts + delta
__device__ __forceinline__ uint32_t tb_contribution(uint32_t reg, int delta, int lo, int hi, int ts, int shc)
{
    uint32_t v = (reg << delta) >> shc;
    v &= ~0u << (lo - ts);
    v &= ~(~0u << (hi - ts));
    return v;
}

// phase B of the traceback: every queued retired path needs NJ more jumps; any lane can run any task (the ring is in
// shared memory), so the warp shares them evenly, two per lane at a time
template <int PACK>
__device__ __noinline__ void tb_run_tasks(const Smem<PACK> sm, int ntask, int ts, int NJ, int shc)
{
    const int lane = threadIdx.x;
    __syncwarp();
    for (int base = 0; base < ntask; base += 2 * BD) {
        Jumper<PACK, uint32_t> tw[2];
        int lo[2], thi[2], dst[2], dl[2];
        bool on[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int i = base + u * BD + lane;
            on[u] = i < ntask;
            const uint2 tk = on[u] ? sm_at<uint2>(sm.tasks + i * 8) : make_uint2(0u, 0u);
            const uint32_t a = tk.x;
            const int col = a & 31, fi = (a >> 5) & 1;
            lo[u] = ts + (int)((a >> 12) & 31u); thi[u] = ts + (int)((a >> 17) & 31u);
            dl[u] = (int)((a >> 22) & 15u) << 2;
            dst[u] = sm.outbits + (col + BD * fi) * 4;
            tw[u].init(sm, (int)((a >> 6) & 63u), col, fi, tk.y);
        }
#pragma unroll 1
        for (int i = 0; i < NJ; ++i) {
#pragma unroll
            for (int u = 0; u < 2; ++u) tw[u].jump();
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            if (!on[u]) continue;
            const uint32_t bits = tb_contribution(tw[u].reg, dl[u], lo[u], thi[u], ts, shc);
            if (bits) atomicOr(&sm_at<uint32_t>(dst[u]), bits);
        }
    }
    __syncwarp();
}

// Traceback of the windows tau in (ts, te] (App. A.1-8): output bit p = tau - D + 1 is the input u_{tau-D+2} on the
// survivor path that starts at best[tau]  (ts is a block boundary; te = ts + TBB, or T in the final block).
//   phase A  every thread walks tau = te .. ts+1 once along the current path of each of its frames (one look-up per
//            B steps); where the path misses best[tau] it is retired into a task (it still owes the bits of the
//            windows (tau, hi] it served) and a new path starts from the field of best[tau].  The whole warp walks in
//            lock step, so task slots come from a ballot -- no atomics.
//   phase B  every retired path needs NJ more jumps; any lane can run any task (the ring is in shared memory), so
//            the warp shares them evenly, two per lane at a time.
// A path that served the windows (lo, hi], was retired in the block above boundary t0s and has been jumped NJ times
// holds block bit k (window ts+1+k) at register bit k + shc - (t0s - ts), shc = 4*NJ - D + 8 in [0, 3].
// In the final block the path from best[T] also owns every later bit up to L-1 (a separate 64-bit walk).
template <class CODE, int PACK>
__device__ __forceinline__ void tb_block_body(const Smem<PACK> sm, int ts, int te, int slot_last, int D, int L, int NJ,
                                               uint8_t *out0, uint8_t *out1, int valid_mask, int out_vec8, bool final)
{
    const int lane = threadIdx.x;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const int p0 = ts - D + 2;                          // output bit of window ts+1
    const int shc = 4 * NJ - D + 8;
    const int jte = (te - 1) & 3;
    // ring slot of the block that ended at the boundary below te
    int bslot0 = slot_last;
    if (jte == 3) bslot0 = (slot_last == 0) ? sm.RB - 1 : slot_last - 1;
    uint32_t acc[PACK];
    Jumper<PACK, uint32_t> jw[PACK];
    int ntask = 0;                                      // warp-uniform
    // best fields of the block that holds te
    int bfo = sm.bf + (((te - 1 - ts) >> 2) * BD + lane) * 16;
    uint4 bq = sm_at<uint4>(bfo);
    const uint32_t bwe = (jte == 0) ? bq.x : (jte == 1) ? bq.y : (jte == 2) ? bq.z : bq.w;
#pragma unroll
    for (int fi = 0; fi < PACK; ++fi) {
        jw[fi].init(sm, bslot0, lane, fi, (bwe >> (16 * fi)) & 0x3FFu);
        sm_at<uint32_t>(sm.outbits + (lane + BD * fi) * 4) = 0u;
    }
    // one window: does the current path of frame fi pass through best[tau]?  (j = sub-step of tau, bw = best fields)
    // Branch free, and the only serial dependency from one window to the next is xor-and -> compare -> select on the
    // path register: the task slot comes from a ballot, the task is stored unconditionally (lanes that do not retire
    // write a scratch slot of their own).
    uint32_t hi_sh[PACK];                               // (hi - ts) << 17, the form the task word wants
#pragma unroll
    for (int fi = 0; fi < PACK; ++fi) hi_sh[fi] = (uint32_t)(te - ts) << 17;
    const int scratch = sm.tasks + (TASK_CAP + lane) * 8;
    // per frame and block of 4 windows: lane | fi << 5 | ring slot of the next jump << 6 | boundary below the block << 22
    // (hoisted out of the per-window work: it changes only at a jump)
    uint32_t tcb[PACK];
    auto block_const = [&](int t0_rel) {
#pragma unroll
        for (int fi = 0; fi < PACK; ++fi)
            tcb[fi] = (uint32_t)lane | ((uint32_t)fi << 5) | (((uint32_t)jw[fi].rowoff / (uint32_t)Jumper<PACK, uint32_t>::ROWB) << 6) |
                      ((uint32_t)(t0_rel >> 2) << 22);
    };
    // tl = tau - ts of the window, as tl12 = tl << 12
    auto check = [&](uint32_t tl12, int j, uint32_t bw) {
        const uint32_t msk = 63u << (j + 1);
#pragma unroll
        for (int fi = 0; fi < PACK; ++fi) {
            const uint32_t b = (bw >> (16 * fi)) & 0x3FFu;
            const bool miss = ((jw[fi].reg ^ b) & msk) != 0u;
            const uint32_t vote = __ballot_sync(0xffffffffu, miss);
            const int qi = ntask + __popc(vote & lt_mask);
            ntask += __popc(vote);
            // retire the path (it served the windows (tau, hi]) and start the one of best[tau]
            sm_at<uint2>(miss ? sm.tasks + qi * 8 : scratch) = make_uint2(tcb[fi] | tl12 | hi_sh[fi], jw[fi].reg);
            hi_sh[fi] = miss ? (tl12 << 5) : hi_sh[fi];
            jw[fi].reg = miss ? b : jw[fi].reg;
        }
    };
    // a block of 4 windows can queue up to 8 * 32 tasks: drain the queue first when that might not fit (rare)
    auto make_room = [&]() {
        if (__builtin_expect(ntask > TASK_CAP - 8 * BD, 0)) {
            tb_run_tasks<PACK>(sm, ntask, ts, NJ, shc);
            ntask = 0;
        }
    };
    // ---- phase A: the rest of the block that holds te, then whole blocks down to ts
    int tau = te - 1;
    block_const(te - 1 - jte - ts);
    for (int j = jte - 1; j >= 0; --j, --tau)
        check((uint32_t)(tau - ts) << 12, j, (j == 0) ? bq.x : (j == 1) ? bq.y : bq.z);
    while (tau > ts) {
        make_room();
#pragma unroll
        for (int fi = 0; fi < PACK; ++fi) jw[fi].jump();
        bfo -= BD * 16;
        bq = sm_at<uint4>(bfo);
        block_const(tau - 4 - ts);
        const uint32_t tl12 = (uint32_t)(tau - ts) << 12;
        check(tl12, 3, bq.w);
        check(tl12 - (1u << 12), 2, bq.z);
        check(tl12 - (2u << 12), 1, bq.y);
        check(tl12 - (3u << 12), 0, bq.x);
        tau -= 4;
    }
    // ---- closing paths of this thread's own frames (interleaved for ILP); the walk above ended at boundary ts
#pragma unroll 1
    for (int i = 0; i < NJ; ++i) {
#pragma unroll
        for (int fi = 0; fi < PACK; ++fi) jw[fi].jump();
    }
#pragma unroll
    for (int fi = 0; fi < PACK; ++fi) acc[fi] = tb_contribution(jw[fi].reg, 0, ts, ts + (int)(hi_sh[fi] >> 17), ts, shc);
    // ---- phase B: the retired paths
    tb_run_tasks<PACK>(sm, ntask, ts, NJ, shc);
#pragma unroll
    for (int fi = 0; fi < PACK; ++fi) {
        const uint32_t a32 = acc[fi] | sm_at<uint32_t>(sm.outbits + (lane + BD * fi) * 4);
        if (!((valid_mask >> fi) & 1)) continue;
        uint8_t *orow = (fi == 0 ? out0 : out1);
        const int nbw = te - ts;
        if (out_vec8 == 2) {
            // bit-packed output (host launcher guarantees p0 % 8 == 0, TBB % 8 == 0, L % 8 == 0): bit p of the frame is
            // bit 7 - (p & 7) of byte p >> 3
            unsigned long long a64 = a32;
            int nb = nbw;
            if (final) {
                Jumper<PACK, unsigned long long> t;
                t.init(sm, bslot0, lane, fi, (unsigned long long)((bwe >> (16 * fi)) & 0x3FFu));
#pragma unroll 1
                for (int i = 0; i < NJ; ++i) t.jump();
                a64 |= (t.reg >> (jte + 1 + shc)) << nbw;          // bits T-D+2 .. L-1 follow the last window
                nb = L - p0;
            }
            for (int g8 = 0; g8 < nb; g8 += 8)
                orow[(p0 + g8) >> 3] = (uint8_t)(__brev((uint32_t)(a64 >> g8) & 0xffu) >> 24);
            continue;
        }
        if (out_vec8 && p0 >= 0 && (p0 & 7) == 0 && (nbw & 7) == 0) {
            // 8 decoded bits -> 8 bytes per store
            for (int g8 = 0; g8 < nbw; g8 += 8) {
                const uint32_t b8 = (a32 >> g8) & 0xffu;
                uint2 v;
                v.x = (((b8 >> 0) & 15u) * 0x00204081u) & 0x01010101u;
                v.y = (((b8 >> 4) & 15u) * 0x00204081u) & 0x01010101u;
                *reinterpret_cast<uint2 *>(orow + p0 + g8) = v;
            }
        } else {
            for (int i = 0; i < nbw; ++i)
                if (p0 + i >= 0) orow[p0 + i] = (uint8_t)((a32 >> i) & 1u);
        }
        if (final) {
            // the path from best[T] decides every bit from T-D+2 on (u_{T-D+3} .. u_{T-5}): D-7 bits
            Jumper<PACK, unsigned long long> t;
            t.init(sm, bslot0, lane, fi, (unsigned long long)((bwe >> (16 * fi)) & 0x3FFu));
#pragma unroll 1
            for (int i = 0; i < NJ; ++i) t.jump();
            const unsigned long long tail = t.reg >> (jte + 1 + shc);
            const int pt = te - D + 2;
            for (int i = 0; i < D - 7 && pt + i < L; ++i) orow[pt + i] = (uint8_t)((tail >> i) & 1ull);
        }
    }
    __syncwarp();
}

// the traceback is a call in the hard kernel (its 64 packed keys stay in callee-saved registers) and inlined in the
// register-capped soft kernel
template <class CODE, int PACK>
__device__ __noinline__ void tb_block_call(const Smem<PACK> sm, int ts, int te, int slot_last, int D, int L, int NJ,
                                           uint8_t *out0, uint8_t *out1, int valid_mask, int out_vec8, bool final)
{
    tb_block_body<CODE, PACK>(sm, ts, te, slot_last, D, L, NJ, out0, out1, valid_mask, out_vec8, final);
}
template <class CODE, int PACK>
__device__ __forceinline__ void tb_block(const Smem<PACK> sm, int ts, int te, int slot_last, int D, int L, int NJ,
                                         uint8_t *out0, uint8_t *out1, int valid_mask, int out_vec8, bool final)
{
    if constexpr (PACK == 1)
        tb_block_body<CODE, PACK>(sm, ts, te, slot_last, D, L, NJ, out0, out1, valid_mask, out_vec8, final);
    else
        tb_block_call<CODE, PACK>(sm, ts, te, slot_last, D, L, NJ, out0, out1, valid_mask, out_vec8, final);
}
constexpr int QD_HARD = 4;         // input prefetch distance of the hard kernel, in pairs of steps
constexpr int QD_SOFT = 2;         // input prefetch distance of the soft kernels, in pairs of steps
constexpr int SOFT_MIN_CTAS = 8;   // __launch_bounds__ minimum CTAs per SM of the soft kernels (12 -- a 168-register cap -- measured 2.7 % slower)
constexpr int TB_DEPHASE = 8;      // windows in the first traceback block of the second warp of a scheduler (0: off)

template <class CODE, int PACK, int QD, int IOP>
__device__ __forceinline__ void viterbi_fast_body(const Params &p)
{
    using OPS = KeyOps<PACK>;
    constexpr int S = CODE::S, M = CODE::M;
    constexpr int NW = 8 * PACK;
    static_assert(S == 64 && M == 6, "fast path is written for 64 states");
    const int tid = threadIdx.x;
    Smem<PACK> sm;
    {
        int q = 0;
        sm.RB = p.RB;
        sm.nib = q; q += p.RB * NW * BD * (int)sizeof(uint32_t);
        sm.bf = q; q += p.TBB * BD * (int)sizeof(uint32_t);
        sm.lut = q; q += 16 * (int)sizeof(uint4);
        sm.tasks = q; q += 2 * (TASK_CAP + BD) * (int)sizeof(uint32_t);
        sm.outbits = q;
    }
    if (PACK == 2) {
        // hard-decision branch metrics of two frames: entry idx = r0A | r1A<<1 | r0B<<2 | r1B<<3,
        // component o = Hamming distance to output symbol o (convcode.py:579) in the metric field, frame B in the high half
        if (tid < 16) {
            // table index: r0A | r1A<<1 | r0B<<2 | r1B<<3 (byte input) or symA | symB<<2 with sym = r0<<1 | r1 (packed input)
            const int a = (IOP == 1) ? (tid & 3) : (((tid & 1) << 1) | ((tid >> 1) & 1));
            const int b = (IOP == 1) ? (tid >> 2) : ((((tid >> 2) & 1) << 1) | ((tid >> 3) & 1));
            uint32_t e[4];
            for (int o = 0; o < 4; ++o) e[o] = ((uint32_t)__popc(o ^ a) << FB) | ((uint32_t)__popc(o ^ b) << (16 + FB));
            sm_at<uint4>(sm.lut + tid * 16) = make_uint4(e[0], e[1], e[2], e[3]);
        }
        __syncwarp();
    }

    // frames of this thread (frame B = frame A + 32)
    const int64_t base = (int64_t)blockIdx.x * BD * PACK;
    int64_t fr[PACK];
    int valid_mask = 0;
    uint8_t *outp[2] = {nullptr, nullptr};
#pragma unroll
    for (int fi = 0; fi < PACK; ++fi) {
        fr[fi] = base + (int64_t)fi * BD + tid;
        if (fr[fi] < p.batch) valid_mask |= 1 << fi; else fr[fi] = p.batch - 1;
        outp[fi] = p.out + fr[fi] * (int64_t)(IOP == 1 ? (p.L >> 3) : p.L);
    }

    // float input: the frame's own power-of-two scale (frame_scale_kernel), so a frame decodes identically
    // whatever it is batched with
    float scale = 1.0f, padq = 0.0f;
    if (PACK == 1) {
        scale = __ldg(p.frame_scale + fr[0]);
        padq = (p.mode == CPB_VITERBI_UNQUANTIZED) ? -1.0f : 0.0f;   // convcode.py:727-732
    }

    uint32_t K[64], Kn[64];
    {
        // pm[0] = 0, every other state "infinite" (convcode.py:705-706): a finite sentinel larger than any
        // metric a path starting in state 0 can lose against (n*M*max branch metric) behaves identically.
        const uint32_t big = (PACK == 2) ? (16u << FB) : ((uint32_t)(13 * QMAX) << FB);
#pragma unroll
        for (int s = 0; s < 64; ++s) {
            const uint32_t v = (s == 0) ? 0u : big;
            K[s] = (PACK == 2) ? ((v | (v << 16)) | OPS::idx(s)) : (v | OPS::idx(s));
        }
    }
    const uint32_t met = p.met_mask;

    const unsigned char *c8 = reinterpret_cast<const unsigned char *>(p.coded);
    const float *cf = reinterpret_cast<const float *>(p.coded);
    const int npairs_in = p.L >> 1;              // pairs of steps fully covered by received data

    // received values of the pair of steps (2 pr + 1, 2 pr + 2)
    //   hard: the 4 coded bytes of frame A and of frame B;  float: the 4 raw values
    struct Raw { uint32_t w[(PACK == 2) ? 2 : 4]; };
    int pc_pos = 0;
    int64_t pc_idx = 0;
    auto load_pair = [&](int pr) {
        Raw r;
        if (PACK == 2) {
            // a = the 4 coded bytes of frame A, b = frame B; past the data: zeros (convcode.py:727-728)
            uint32_t a = 0u, b = 0u;
            if (IOP == 1) {
                // bit-packed input: the byte that holds the pair (2 pairs of steps per byte, first element in bit 7)
                if (pr < npairs_in) {
                    a = __ldg(c8 + fr[0] * (p.n_in >> 3) + (pr >> 1));
                    b = __ldg(c8 + fr[PACK - 1] * (p.n_in >> 3) + (pr >> 1));
                }
            } else if (p.in_aligned && pr < npairs_in) {
                a = __ldg(reinterpret_cast<const uint32_t *>(c8 + fr[0] * p.n_in) + pr);
                b = __ldg(reinterpret_cast<const uint32_t *>(c8 + fr[PACK - 1] * p.n_in) + pr);
            } else {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int tau = 2 * pr + 1 + h;
                    if (tau <= p.L) {
                        const unsigned char *qa = c8 + fr[0] * p.n_in + 2 * (int64_t)(tau - 1);
                        const unsigned char *qb = c8 + fr[PACK - 1] * p.n_in + 2 * (int64_t)(tau - 1);
                        a |= ((uint32_t)__ldg(qa) | ((uint32_t)__ldg(qa + 1) << 8)) << (16 * h);
                        b |= ((uint32_t)__ldg(qb) | ((uint32_t)__ldg(qb + 1) << 8)) << (16 * h);
                    }
                }
            }
            r.w[0] = a; r.w[1] = b;         // (nothing is computed here: the queue must not wait for the load)
        } else {
            const uint32_t pb = __float_as_uint(padq);
            r.w[0] = r.w[1] = r.w[2] = r.w[3] = pb;
            const float *row = cf + fr[0] * (IOP == 2 ? p.n_kept : p.n_in);
            if (IOP == 2) {
                // depuncturing fused into the load: the queue asks for the pairs in order, so the position in the
                // puncturing period and in the punctured row are running counters
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                    if (2 * pr + 1 + (h >> 1) <= p.L) {
                        float v = 0.0f;                                  // erased position (convcode.py:796-799)
                        if ((p.punct_mask >> pc_pos) & 1u) { v = __ldg(row + pc_idx); ++pc_idx; }
                        pc_pos = (pc_pos + 1 == p.punct_len) ? 0 : pc_pos + 1;
                        r.w[h] = __float_as_uint(v);
                    }
                }
            } else if (p.in_aligned && pr < npairs_in) {
                const float4 v = __ldg(reinterpret_cast<const float4 *>(row) + pr);
                r.w[0] = __float_as_uint(v.x); r.w[1] = __float_as_uint(v.y); r.w[2] = __float_as_uint(v.z); r.w[3] = __float_as_uint(v.w);
            } else {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int tau = 2 * pr + 1 + h;
                    if (tau <= p.L) {
                        r.w[2 * h] = __float_as_uint(__ldg(row + 2 * (int64_t)(tau - 1)));
                        r.w[2 * h + 1] = __float_as_uint(__ldg(row + 2 * (int64_t)(tau - 1) + 1));
                    }
                }
            }
        }
        return r;
    };
    // hard: the 4 received bits of a step (two frames) are gathered into one nibble by two multiplies.  Bytes (r0, r1 of
    // step a, r0, r1 of step b), each 0/1 -> bits (0,1,4,5) [frame A] / (2,3,6,7) [frame B] of the top byte: term
    // 2^(24-8i+pos_i) moves byte i to bit 24+pos_i, every stray product lands on its own lower bit (no carries).
    // Byte (w >> 24) = table index of step a | table index of step b << 4.
    auto gather = [&](const Raw &r) {
        Raw g = r;
        if (PACK == 2 && IOP != 1) g.w[0] = (r.w[0] & 0x01010101u) * 0x01021020u + (r.w[1] & 0x01010101u) * 0x04084080u;
        return g;
    };
    // the four branch metrics (in the metric field) of step h (0 / 1) of a (gathered) pair
    // (bit-packed input: `odd` says whether the pair is the second one of its byte)
    auto make_bm = [&](const Raw &r, int h, uint32_t (&Bm)[4], int odd = 0) {
        if (PACK == 2 && IOP == 1) {
            // received symbol of frame A = bits (7,6) >> 2*(2*odd + h) of its byte, same for frame B; table index = A | B << 2
            const int sh = 2 * (2 * odd + h);
            const uint32_t off = (((r.w[0] << sh) >> 2) & 0x30u) | ((r.w[1] << sh) & 0xC0u);
            const uint4 e = sm_at<uint4>(sm.lut + (int)off);
            Bm[0] = e.x; Bm[1] = e.y; Bm[2] = e.z; Bm[3] = e.w;
        } else if (PACK == 2) {
            const uint32_t off = (r.w[0] >> (h ? 24 : 20)) & 0xF0u;      // 16 * table index
            const uint4 e = sm_at<uint4>(sm.lut + (int)off);
            Bm[0] = e.x; Bm[1] = e.y; Bm[2] = e.z; Bm[3] = e.w;
        } else {
            float r0 = __uint_as_float(r.w[2 * h]), r1 = __uint_as_float(r.w[2 * h + 1]);
            if (p.mode == CPB_VITERBI_SOFT) {          // convcode.py:718-719
                r0 = fminf(fmaxf(r0, -500.0f), 500.0f);
                r1 = fminf(fmaxf(r1, -500.0f), 500.0f);
            }
            const int q0 = __float2int_rn(fminf(fmaxf(r0 * scale, -(float)QMAX), (float)QMAX));
            const int q1 = __float2int_rn(fminf(fmaxf(r1 * scale, -(float)QMAX), (float)QMAX));
            // -log-likelihood of code bit c given value r, up to a per-step constant (convcode.py:581-587):
            // c = 0 costs max(q,0), c = 1 costs max(-q,0)
            const uint32_t z0 = (uint32_t)max(q0, 0) << FB, o0 = (uint32_t)max(-q0, 0) << FB;
            const uint32_t z1 = (uint32_t)max(q1, 0) << FB, o1 = (uint32_t)max(-q1, 0) << FB;
            Bm[0] = z0 + z1; Bm[1] = z0 + o1; Bm[2] = o0 + z1; Bm[3] = o0 + o1;
        }
    };

    const int ts0 = (p.D - 2) & ~3;              // first traceback block starts at this boundary (windows exist from D-1)
    int ts_cur = ts0;
    int next_te = ts_cur + p.TBB;
    if (TB_DEPHASE) {
        // The traceback is latency bound, the add-compare-select loop pipe bound: two warps that share a scheduler
        // (hardware warp slots w and w+4) should not trace back at the same time, so the second one ends its first
        // traceback block half a period early.  (Scheduling only: the output does not depend on the block boundaries.)
        uint32_t wid;
        asm("mov.u32 %0, %%warpid;" : "=r"(wid));
        if ((wid >> 2) & 1u) next_te = ts_cur + TB_DEPHASE;   // a multiple of 8: output stores stay 8-byte aligned
    }
    int nslot = 0;                               // ring slot the next completed block goes to

    // end of a block of B steps (keys in Kc, mn = minimum key of the last step): jump nibbles to the ring, keys back to
    // metric | state, renormalisation
    auto block_end = [&](uint32_t (&Kc)[64], uint32_t mn, int tau) {
        const int nb = sm.nib + (nslot * NW * BD + tid) * 4;
        if (PACK == 2) {
#pragma unroll
            for (int w = 0; w < 16; ++w) {
                const uint32_t t0 = (Kc[4 * w] & OPS::NIBM) | ((Kc[4 * w + 1] << 4) & ~OPS::NIBM);
                const uint32_t t1 = (Kc[4 * w + 2] & OPS::NIBM) | ((Kc[4 * w + 3] << 4) & ~OPS::NIBM);
                sm_at<uint32_t>(nb + w * BD * 4) = __byte_perm(t0, t1, 0x6240);
            }
        } else {
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                uint32_t t[4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    t[i] = (Kc[8 * w + 2 * i] & OPS::NIBM) | ((Kc[8 * w + 2 * i + 1] << 4) & ~OPS::NIBM);
                sm_at<uint32_t>(nb + w * BD * 4) =
                    __byte_perm(__byte_perm(t[0], t[1], 0x0040), __byte_perm(t[2], t[3], 0x0040), 0x5410);
            }
        }
        // renormalisation: every block for the 22-bit float metrics; every 16 steps for the 6-bit Hamming metrics
        // (spread <= 12, growth <= 2 per step: 12 + 32 + 2 < 64)
        if (PACK == 1) {
            const uint32_t sub = mn & ~OPS::FMASK;
#pragma unroll
            for (int s = 0; s < 64; ++s) Kc[s] = ((Kc[s] & met) | OPS::idx(s)) - sub;
        } else {
#pragma unroll
            for (int s = 0; s < 64; ++s) Kc[s] = (Kc[s] & met) | OPS::idx(s);
            if ((tau & 15) == 0) {
                const uint32_t sub = mn & ~OPS::FMASK;
#pragma unroll
                for (int s = 0; s < 64; ++s) Kc[s] -= sub;
            }
        }
    };

    Raw qd[QD];
#pragma unroll
    for (int i = 0; i < QD; ++i) qd[i] = load_pair(i);
    uint32_t Bm[4];
    uint32_t mq0 = 0u, mq1 = 0u;                 // best fields of the first half of the running block
    static_assert(QD >= 2 && QD % 2 == 0, "the prefetch queue moves by whole blocks");
    const int npairs = p.T >> 1, nfull = p.T >> 2;
    // (A loop body of half a block -- smaller code -- was measured: slower, the register shuffling at the extra loop
    // edge costs more than the instruction fetch it saves.)
#pragma unroll 1
    for (int blk = 0; blk < nfull; ++blk) {
        const Raw cur0 = gather(qd[0]), cur1 = gather(qd[1]);
#pragma unroll
        for (int i = 0; i + 2 < QD; ++i) qd[i] = qd[i + 2];
        qd[QD - 2] = load_pair(2 * blk + QD);          // software prefetch, QD pairs of steps ahead
        qd[QD - 1] = load_pair(2 * blk + QD + 1);
        make_bm(cur0, 0, Bm);
        mq0 = acs_step<CODE, PACK>(K, Kn, Bm, OPS::INC0 << 0);
        make_bm(cur0, 1, Bm);
        mq1 = acs_step<CODE, PACK>(Kn, K, Bm, OPS::INC0 << 1);
        make_bm(cur1, 0, Bm, 1);
        const uint32_t m2 = acs_step<CODE, PACK>(K, Kn, Bm, OPS::INC0 << 2);
        make_bm(cur1, 1, Bm, 1);
        const uint32_t m3 = acs_step<CODE, PACK>(Kn, K, Bm, OPS::INC0 << 3);
        const int tau = 4 * blk + 4, tau0 = 4 * blk;
        if (tau0 >= ts_cur)
            sm_at<uint4>(sm.bf + (((tau0 - ts_cur) >> 2) * BD + tid) * 16) =
                make_uint4(mq0 & OPS::FMASK, mq1 & OPS::FMASK, m2 & OPS::FMASK, m3 & OPS::FMASK);
        block_end(K, m3, tau);
        if (tau == next_te || tau == p.T) {
            tb_block<CODE, PACK>(sm, ts_cur, tau, nslot, p.D, p.L, p.NJ, outp[0], outp[PACK - 1], valid_mask, p.out_vec8, tau == p.T);
            ts_cur = tau;
            next_te = tau + p.TBB;
        }
        nslot = (nslot + 1 == p.RB) ? 0 : nslot + 1;
    }
    mq0 = mq1 = 0u;
    if (npairs & 1) {                            // T mod 4 >= 2: one more pair of steps
        const Raw cur = gather(qd[0]);
        make_bm(cur, 0, Bm);
        mq0 = acs_step<CODE, PACK>(K, Kn, Bm, OPS::INC0) & OPS::FMASK;
        make_bm(cur, 1, Bm);
        mq1 = acs_step<CODE, PACK>(Kn, K, Bm, OPS::INC0 << 1) & OPS::FMASK;
        qd[0] = qd[1];
    }
    if (p.T & 3) {
        // the last 1..3 steps: no block completes, the final traceback starts from best[T]'s field
        uint32_t mq2 = 0u;
        if (p.T & 1) {
            make_bm(gather(qd[0]), 0, Bm, npairs & 1);
            const uint32_t m = acs_step<CODE, PACK>(K, Kn, Bm, OPS::INC0 << (2 * (npairs & 1))) & OPS::FMASK;
            if (npairs & 1) mq2 = m; else mq0 = m;
        }
        const int tau0 = p.T & ~3;
        sm_at<uint4>(sm.bf + (((tau0 - ts_cur) >> 2) * BD + tid) * 16) = make_uint4(mq0, mq1, mq2, 0u);
        const int last = (nslot == 0) ? p.RB - 1 : nslot - 1;
        tb_block<CODE, PACK>(sm, ts_cur, p.T, last, p.D, p.L, p.NJ, outp[0], outp[PACK - 1], valid_mask, p.out_vec8, true);
    }
}

// hard decision: two u16x2-packed frames per thread
template <class CODE>
__global__ void __launch_bounds__(BD) viterbi_fast_kernel_hard(const Params p) { viterbi_fast_body<CODE, 2, QD_HARD, 0>(p); }
// the same with bit-packed input and output (1 bit per coded / decoded bit, np.packbits order): 8x less HBM and PCIe traffic
template <class CODE>
__global__ void __launch_bounds__(BD) viterbi_fast_kernel_hard_packed(const Params p) { viterbi_fast_body<CODE, 2, QD_HARD, 1>(p); }
// soft / unquantized: one frame per thread, 32-bit keys
template <class CODE>
__global__ void __launch_bounds__(BD, SOFT_MIN_CTAS) viterbi_fast_kernel_soft(const Params p) { viterbi_fast_body<CODE, 1, QD_SOFT, 0>(p); }
// the same on punctured rows: depuncturing (convcode.py:777-804) happens in the load
template <class CODE>
__global__ void __launch_bounds__(BD, SOFT_MIN_CTAS) viterbi_fast_kernel_soft_punct(const Params p) { viterbi_fast_body<CODE, 1, QD_SOFT, 2>(p); }

// Per-frame power-of-two scale for float input: the largest |value| of the frame (after the +-500 clip in 'soft'
// mode, convcode.py:718-719; including the -1 padding of 'unquantized', :729-732) maps to at most 2^QBITS.
// One warp per frame, coalesced; a frame's scale depends on nothing but the frame.
__global__ void frame_scale_kernel(const float *__restrict__ x, int64_t n_in, int64_t n_used, int64_t batch, int mode,
                                   float *__restrict__ scale)
{
    const int64_t f = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (f >= batch) return;
    const int lane = threadIdx.x & 31;
    const float *row = x + f * n_in;
    float m = (mode == CPB_VITERBI_UNQUANTIZED) ? 1.0f : 0.0f;
    auto take = [&](float v) {
        v = fabsf(v);
        if (!(v <= 3.0e38f)) v = 3.0e38f;      // inf / nan
        if (mode == CPB_VITERBI_SOFT) v = fminf(v, 500.0f);
        m = fmaxf(m, v);
    };
    if ((n_in & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) & 15) == 0)) {
        const float4 *r4 = reinterpret_cast<const float4 *>(row);
        const int64_t n4 = n_used >> 2;
        for (int64_t i = lane; i < n4; i += 32) { const float4 v = __ldg(r4 + i); take(v.x); take(v.y); take(v.z); take(v.w); }
        for (int64_t i = (n4 << 2) + lane; i < n_used; i += 32) take(__ldg(row + i));
    } else {
        for (int64_t i = lane; i < n_used; i += 32) take(__ldg(row + i));
    }
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) {
        m = fminf(fmaxf(m, 1e-30f), 3.0e38f);
        float s = exp2f(floorf(log2f((float)QMAX / m)));
        if (m * s > (float)QMAX) s *= 0.5f;     // log2f rounding at exact powers of two
        scale[f] = fminf(s, 1.0e30f);
    }
}

template <class CODE, int PACK, int IOP>
static int launch(const Params &p, cudaStream_t st)
{
    const size_t smem = smem_bytes(p.RB, p.TBB, PACK);
    void (*kern)(const Params) = (IOP == 1) ? viterbi_fast_kernel_hard_packed<CODE>
                               : (IOP == 2) ? viterbi_fast_kernel_soft_punct<CODE>
                               : (PACK == 2) ? viterbi_fast_kernel_hard<CODE> : viterbi_fast_kernel_soft<CODE>;
    { const int rc_ = ensure_dyn_smem(reinterpret_cast<const void *>(kern), smem); if (rc_) return rc_; }
    const int64_t grid = ceil_div(p.batch, (int64_t)BD * PACK);
    kern<<<(unsigned)grid, BD, smem, st>>>(p);
    CPB_LAUNCH_CHECK();
    return CPB_OK;
}

}  // namespace fast

// ------------------------------------------------------------------------------------------------
// Generic table-driven path
// ------------------------------------------------------------------------------------------------
namespace gen {

constexpr int BD = 64;
constexpr int TBB = 32;

struct Params {
    const void *coded;
    int in_dtype;
    int64_t n_in;
    int64_t frame0;       // first frame of this chunk
    int nframes;          // frames in this chunk
    int64_t stride;       // frame stride of the scratch planes (>= nframes)
    const int32_t *pred;
    int k, n, S, I;
    int L, T, D, mode;
    uint8_t *winners;     // [(T+1)*S][stride]
    uint8_t *best;        // [T+1][stride]
    uint8_t *out;
};

__global__ void __launch_bounds__(BD) viterbi_generic_kernel(const Params p)
{
    extern __shared__ float sm[];
    const int tid = threadIdx.x;
    const int S = p.S, I = p.I, n = p.n, k = p.k;
    const int NB = 1 << n;
    float *pm0 = sm;                       // [S][BD]
    float *pm1 = sm + (size_t)S * BD;      // [S][BD]
    float *bmv = sm + (size_t)2 * S * BD;  // [NB][BD]
    const int f = blockIdx.x * BD + tid;
    const bool valid = f < p.nframes;
    const int64_t frame = p.frame0 + (valid ? f : 0);
    const unsigned char *c8 = reinterpret_cast<const unsigned char *>(p.coded) + frame * p.n_in;
    const float *cf = reinterpret_cast<const float *>(p.coded) + frame * p.n_in;
    const int64_t fcol = valid ? f : 0;

    for (int s = 0; s < S; ++s) pm0[s * BD + tid] = (s == 0) ? 0.0f : INFINITY;     // convcode.py:705-706
    float *po = pm0, *pn = pm1;
    const int64_t Lk = p.L / k;
    const float padv = (p.mode == CPB_VITERBI_UNQUANTIZED) ? -1.0f : 0.0f;

    for (int tau = 1; tau <= p.T; ++tau) {
        float r[4];
        for (int j = 0; j < n; ++j) {
            float v = padv;
            if (tau <= Lk) {
                const int64_t e = (int64_t)(tau - 1) * n + j;
                v = (p.in_dtype == CPB_U8) ? (float)(c8[e] & 1u) : cf[e];
            }
            if (p.mode == CPB_VITERBI_SOFT) v = fminf(fmaxf(v, -500.0f), 500.0f);
            r[j] = v;
        }
        for (int c = 0; c < NB; ++c) {
            float acc = 0.0f;
            for (int j = 0; j < n; ++j) {
                const int cj = (c >> (n - 1 - j)) & 1;           // MSB first
                if (p.mode == CPB_VITERBI_HARD) acc += (((int)r[j]) ^ cj) ? 1.0f : 0.0f;
                else if (p.mode == CPB_VITERBI_SOFT) acc += cj ? fmaxf(-r[j], 0.0f) : fmaxf(r[j], 0.0f);
                else { const float d = r[j] - (float)(2 * cj - 1); acc += d * d; }
            }
            bmv[c * BD + tid] = acc;
        }
        float mn = INFINITY; int arg = 0;
        for (int s = 0; s < S; ++s) {
            float bestm = 0.0f; int bi = 0;
            for (int i = 0; i < I; ++i) {
                const int e = __ldg(&p.pred[s * I + i]);
                const float m = po[(e & 0xff) * BD + tid] + bmv[((e >> 16) & 0xff) * BD + tid];
                if (i == 0 || m < bestm) { bestm = m; bi = i; }
            }
            pn[s * BD + tid] = bestm;
            if (valid) p.winners[((int64_t)tau * S + s) * p.stride + fcol] = (uint8_t)bi;
            if (s == 0 || bestm < mn) { mn = bestm; arg = s; }
        }
        if (valid) p.best[(int64_t)tau * p.stride + fcol] = (uint8_t)arg;
        if (mn < INFINITY && mn != 0.0f)
            for (int s = 0; s < S; ++s) pn[s * BD + tid] -= mn;     // exact for the integer metrics of 'hard'
        float *t_ = po; po = pn; pn = t_;
    }
    if (!valid) return;

    // traceback: symbol of step q comes from the path started at best[min(q + D - 2, T)]
    uint8_t *o = p.out + frame * (int64_t)p.L;
    auto emit = [&](int q, int u) {
        for (int b = 0; b < k; ++b) {
            const int64_t pos = (int64_t)(q - 1) * k + b;
            if (pos < p.L) o[pos] = (uint8_t)((u >> (k - 1 - b)) & 1);
        }
    };
    auto prev = [&](int tau, int s, int &u) {
        const int i = p.winners[((int64_t)tau * S + s) * p.stride + fcol];
        const int e = __ldg(&p.pred[s * I + i]);
        u = (e >> 8) & 0xff;
        return e & 0xff;
    };
    auto bestat = [&](int tau) { return (int)p.best[(int64_t)tau * p.stride + fcol]; };

    int ts = p.D - 2;
    while (ts < p.T) {
        int te = ts + TBB;
        bool fin = false;
        if (te >= p.T) { te = p.T; fin = true; }
        int s = bestat(te);
        uint32_t cons = 0;
        const int tau_min = max(1, ts - p.D + 3);
        for (int tau = te; tau >= tau_min; --tau) {
            if (tau > ts && s == bestat(tau)) cons |= 1u << (tau - ts - 1);
            int u;
            const int pr = prev(tau, s, u);
            if (fin || tau <= te - p.D + 2) emit(tau, u);
            s = pr;
        }
        for (int tp = ts + 1; tp < te; ++tp) {
            if ((cons >> (tp - ts - 1)) & 1u) continue;
            int s2 = bestat(tp), u = 0;
            for (int tau = tp; tau >= tp - p.D + 2; --tau) {
                if (tau < 1) break;
                s2 = prev(tau, s2, u);
            }
            if (tp - p.D + 2 >= 1) emit(tp - p.D + 2, u);
        }
        ts = te;
    }
}

}  // namespace gen

// ------------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int cpb_trellis_create(const int32_t *next_state, const int32_t *output, int k, int n, int total_memory,
                       int number_states, cpbTrellis **out)
{
    if (!next_state || !output || !out || k < 1 || k > 4 || n < 1 || n > 4 || number_states < 1 ||
        number_states > 256 || total_memory < 0)
        return CPB_EINVAL;
    cpbTrellis *t = new cpbTrellis();
    t->k = k; t->n = n; t->M = total_memory; t->S = number_states; t->I = 1 << k;
    const int S = t->S, I = t->I;
    t->next_state.assign(next_state, next_state + S * I);
    t->output.assign(output, output + S * I);
    std::vector<int32_t> pred(S * I, 0), cnt(S, 0);
    for (int p = 0; p < S; ++p)
        for (int u = 0; u < I; ++u) {
            const int s = next_state[p * I + u], o = output[p * I + u];
            if (s < 0 || s >= S || o < 0 || o >= (1 << n) || cnt[s] >= I) { delete t; return CPB_ETRELLIS; }
            pred[s * I + cnt[s]++] = p | (u << 8) | (o << 16);     // (p asc, u asc): convcode.py:561-572
        }
    for (int s = 0; s < S; ++s)
        if (cnt[s] != I) { delete t; return CPB_ETRELLIS; }
    cudaGetDevice(&t->device);
    const size_t bytes = sizeof(int32_t) * S * I;
    if (cudaMalloc(&t->pred_dev, bytes) != cudaSuccess || cudaMalloc(&t->next_dev, bytes) != cudaSuccess ||
        cudaMalloc(&t->out_dev, bytes) != cudaSuccess) {
        record_cuda_error(cudaGetLastError(), "cudaMalloc(trellis tables)", __FILE__, __LINE__);
        cpb_trellis_destroy(t);
        return CPB_ECUDA;
    }
    cudaMemcpy(t->pred_dev, pred.data(), bytes, cudaMemcpyHostToDevice);
    cudaMemcpy(t->next_dev, t->next_state.data(), bytes, cudaMemcpyHostToDevice);
    cudaError_t e = cudaMemcpy(t->out_dev, t->output.data(), bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        record_cuda_error(e, "cudaMemcpy(trellis tables)", __FILE__, __LINE__);
        cpb_trellis_destroy(t);
        return CPB_ECUDA;
    }
    if (code_matches<Code133_171>(*t)) t->fast_id = 1;
    else if (code_matches<Code171_133>(*t)) t->fast_id = 2;
    else if (code_matches<Code5_43>(*t)) t->fast_id = 3;
    else if (code_matches<Code5_7>(*t)) t->fast_id = 4;
    *out = t;
    return CPB_OK;
}

int cpb_trellis_destroy(cpbTrellis *t)
{
    if (!t) return CPB_OK;
    if (t->pred_dev) cudaFree(t->pred_dev);
    if (t->next_dev) cudaFree(t->next_dev);
    if (t->out_dev) cudaFree(t->out_dev);
    delete t;
    return CPB_OK;
}

int cpb_trellis_fast_path(const cpbTrellis *t) { return t ? t->fast_id : 0; }

}  // extern "C"

// tables for the BCJR kernels (bcjr.cu)
const int32_t *cpb_trellis_next_dev(const cpbTrellis *t) { return t->next_dev; }
const int32_t *cpb_trellis_out_dev(const cpbTrellis *t) { return t->out_dev; }
const int32_t *cpb_trellis_pred_dev(const cpbTrellis *t) { return t->pred_dev; }
void cpb_trellis_dims(const cpbTrellis *t, int *k, int *n, int *S) { *k = t->k; *n = t->n; *S = t->S; }
void cpb_trellis_host_tables(const cpbTrellis *t, const int32_t **next, const int32_t **out)
{
    *next = t->next_state.data();
    *out = t->output.data();
}

static int resolve_depth(const cpbTrellis *t, int64_t L, int tb_depth)
{
    if (tb_depth <= 0) {
        int64_t d = 5 * (int64_t)t->M;          // convcode.py:701-702
        if (d > L) d = L;
        return (int)d;
    }
    return tb_depth;
}

static bool use_fast(const cpbTrellis *t, int D, int mode, int in_dtype)
{
    if (t->fast_id == 0) return false;
    // cpb_set_option(CPB_OPT_VITERBI_FORCE_GENERIC, 1) routes every trellis through the table-driven kernel, so the two
    // independent implementations can be compared against each other at full size (tests/test_viterbi_gpu.py)
    if (option(CPB_OPT_VITERBI_FORCE_GENERIC)) return false;
    if (D < t->M + 1 || D > fast::DMAX) return false;
    if (mode == CPB_VITERBI_HARD) return in_dtype == CPB_U8;
    return in_dtype == CPB_F32;
}

static size_t generic_chunk(const cpbTrellis *t, int64_t batch, int64_t T, int64_t *stride)
{
    // survivors: (T+1)*(S+1) bytes per frame; keep one chunk under ~1.5 GB
    const double per_frame = (double)(T + 1) * (t->S + 1);
    int64_t chunk = (int64_t)(1.5e9 / per_frame);
    chunk = (chunk / gen::BD) * gen::BD;
    if (chunk < gen::BD) chunk = gen::BD;
    const int64_t need = ceil_div(batch, gen::BD) * gen::BD;
    if (chunk > need) chunk = need;
    *stride = chunk;
    return (size_t)((T + 1) * (int64_t)(t->S + 1) * chunk);
}

template <int PACK, int IOP>
static int launch_fast(const cpbTrellis *t, const fast::Params &p, cudaStream_t st)
{
    switch (t->fast_id) {
    case 1: return fast::launch<Code133_171, PACK, IOP>(p, st);
    case 2: return fast::launch<Code171_133, PACK, IOP>(p, st);
    case 3: return fast::launch<Code5_43, PACK, IOP>(p, st);
    default: return fast::launch<Code5_7, PACK, IOP>(p, st);
    }
}

// the launch parameters every fast-path entry point sets alike; CPB_EUNSUPPORTED when the traceback ring does not fit in
// shared memory
static int fast_params(fast::Params &p, const void *coded, int64_t n_in, int64_t batch, int64_t L, int64_t T, int D,
                       int mode, uint8_t *out)
{
    const int pack = (mode == CPB_VITERBI_HARD) ? 2 : 1;
    p.coded = coded; p.n_in = n_in; p.batch = batch;
    p.L = (int)L; p.T = (int)T; p.D = D;
    p.TBB = fast::TBB;
    p.NJ = (D > 8) ? (D - 8 + fast::B - 1) / fast::B : 0;
    p.RB = p.NJ + p.TBB / fast::B;
    p.mode = mode; p.out = out;
    p.out_vec8 = ((L % 8) == 0 && (((uintptr_t)out) % 8) == 0) ? 1 : 0;
    p.met_mask = (pack == 2) ? ~fast::KeyOps<2>::FMASK : ~fast::KeyOps<1>::FMASK;
    return (fast::smem_bytes(p.RB, p.TBB, pack) > device_props().smem_optin) ? CPB_EUNSUPPORTED : CPB_OK;
}

// float input: the power-of-two scale of every frame (over the first n_used values of its row) into the workspace, past
// its first 256 bytes
static int frame_scales(fast::Params &p, const float *x, int64_t n_in, int64_t n_used, void *ws, cudaStream_t st)
{
    float *sc = reinterpret_cast<float *>(reinterpret_cast<unsigned char *>(ws) + 256);
    p.frame_scale = sc;
    const int wpb = 8;
    fast::frame_scale_kernel<<<(unsigned)ceil_div(p.batch, wpb), wpb * 32, 0, st>>>(x, n_in, n_used, p.batch, p.mode, sc);
    const cudaError_t e = cudaGetLastError();
    return (e == cudaSuccess) ? CPB_OK : record_cuda_error(e, "frame_scale_kernel", __FILE__, __LINE__);
}

extern "C" {

int cpb_viterbi_sizes(const cpbTrellis *t, int64_t n_in, int64_t *L, int64_t *T)
{
    if (!t || n_in < 0) return CPB_EINVAL;
    const int64_t l = (int64_t)((double)n_in * ((double)t->k / (double)t->n));      // convcode.py:699
    if (L) *L = l;
    if (T) *T = (int64_t)((double)(l + t->M) / (double)t->k) - 1;                   // :721
    return CPB_OK;
}

int cpb_viterbi_workspace_bytes(const cpbTrellis *t, int64_t batch, int64_t n_in, int tb_depth, int mode, size_t *bytes)
{
    if (!t || !bytes || batch < 0) return CPB_EINVAL;
    int64_t L, T;
    cpb_viterbi_sizes(t, n_in, &L, &T);
    const int D = resolve_depth(t, L, tb_depth);
    const int in_dtype = (mode == CPB_VITERBI_HARD) ? CPB_U8 : CPB_F32;
    if (use_fast(t, D, mode, in_dtype)) { *bytes = 256 + (mode == CPB_VITERBI_HARD ? 0 : (size_t)batch * sizeof(float)); return CPB_OK; }
    int64_t stride;
    *bytes = generic_chunk(t, batch, T, &stride) + 256;
    return CPB_OK;
}

int cpb_viterbi_decode(const cpbTrellis *t, const void *coded_dev, int in_dtype, int64_t batch, int64_t n_in,
                       int tb_depth, int mode, uint8_t *out_bits_dev, void *workspace_dev, size_t workspace_bytes,
                       void *stream)
{
    if (mode < 0 || mode > 2) return CPB_EINVAL;        // ValueError of convcode.py:682-685
    if (t && batch == 0) return CPB_OK;                 // empty tensors carry null pointers
    if (!t || !coded_dev || !out_bits_dev || batch < 0 || n_in < 0) return CPB_EINVAL;
    if (in_dtype != CPB_U8 && in_dtype != CPB_F32) return CPB_EINVAL;
    if (mode != CPB_VITERBI_HARD && in_dtype != CPB_F32) return CPB_EINVAL;
    if (batch == 0) return CPB_OK;
    int64_t L, T;
    cpb_viterbi_sizes(t, n_in, &L, &T);
    const int D = resolve_depth(t, L, tb_depth);
    // the reference returns uninitialised memory when no traceback window ever closes (T < D-1) or D < 2
    if (L <= 0 || D < 2 || T < D - 1 || T > (1 << 24)) return CPB_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;

    if (use_fast(t, D, mode, in_dtype)) {
        const bool hard = (mode == CPB_VITERBI_HARD);
        Scratch ws;
        int rc = ws.acquire(workspace_dev, workspace_bytes, 256 + (hard ? 0 : (size_t)batch * sizeof(float)), st);
        if (rc) return rc;
        fast::Params p{};
        rc = fast_params(p, coded_dev, n_in, batch, L, T, D, mode, out_bits_dev);
        p.in_aligned = ((n_in % 4) == 0 && (((uintptr_t)coded_dev) % (hard ? 4 : 16)) == 0) ? 1 : 0;
        if (!rc && !hard) rc = frame_scales(p, reinterpret_cast<const float *>(coded_dev), n_in, 2 * L, ws.ptr, st);
        if (!rc) rc = hard ? launch_fast<2, 0>(t, p, st) : launch_fast<1, 0>(t, p, st);
        ws.release();
        return rc;
    }

    // generic path, chunked so the survivor scratch stays bounded
    int64_t stride = 0;
    const size_t need = generic_chunk(t, batch, T, &stride);
    Scratch ws;
    int rc = ws.acquire(workspace_dev, workspace_bytes, need, st);
    if (rc) return rc;
    const size_t smem = sizeof(float) * ((size_t)2 * t->S + (1u << t->n)) * gen::BD;
    if (smem > device_props().smem_optin) { ws.release(); return CPB_EUNSUPPORTED; }
    { const int rc_ = ensure_dyn_smem(reinterpret_cast<const void *>(gen::viterbi_generic_kernel), smem); if (rc_) { ws.release(); return rc_; } }
    cudaError_t e = cudaSuccess;
    for (int64_t f0 = 0; f0 < batch; f0 += stride) {
        gen::Params p{};
        p.coded = coded_dev; p.in_dtype = in_dtype; p.n_in = n_in; p.frame0 = f0;
        p.nframes = (int)std::min<int64_t>(stride, batch - f0);
        p.stride = stride; p.pred = t->pred_dev;
        p.k = t->k; p.n = t->n; p.S = t->S; p.I = t->I;
        p.L = (int)L; p.T = (int)T; p.D = D; p.mode = mode;
        p.winners = reinterpret_cast<uint8_t *>(ws.ptr);
        p.best = p.winners + (size_t)(T + 1) * t->S * stride;
        p.out = out_bits_dev;
        gen::viterbi_generic_kernel<<<(unsigned)ceil_div(p.nframes, gen::BD), gen::BD, smem, st>>>(p);
        e = cudaGetLastError();
        if (e != cudaSuccess) { ws.release(); return record_cuda_error(e, "viterbi_generic_kernel", __FILE__, __LINE__); }
    }
    ws.release();
    return CPB_OK;
}


int cpb_viterbi_decode_packed(const cpbTrellis *t, const uint8_t *coded_packed_dev, int64_t batch, int64_t n_in,
                              int tb_depth, uint8_t *out_packed_dev, void *stream)
{
    if (t && batch == 0) return CPB_OK;
    if (!t || !coded_packed_dev || !out_packed_dev || batch < 0 || n_in <= 0) return CPB_EINVAL;
    int64_t L, T;
    cpb_viterbi_sizes(t, n_in, &L, &T);
    const int D = resolve_depth(t, L, tb_depth);
    if (L <= 0 || D < 2 || T < D - 1 || T > (1 << 24)) return CPB_EINVAL;
    // whole bytes per row, whole output bytes per traceback block (fast::TBB % 8 == 0)
    if (!use_fast(t, D, CPB_VITERBI_HARD, CPB_U8) || (n_in % 8) != 0 || (L % 8) != 0 || ((D - 2) % 4) != 0)
        return CPB_EUNSUPPORTED;
    fast::Params p{};
    const int rc = fast_params(p, coded_packed_dev, n_in, batch, L, T, D, CPB_VITERBI_HARD, out_packed_dev);
    if (rc) return rc;
    p.out_vec8 = 2;
    return launch_fast<2, 1>(t, p, (cudaStream_t)stream);
}


int cpb_viterbi_punctured_workspace_bytes(int64_t batch, size_t *bytes)
{
    if (!bytes || batch < 0) return CPB_EINVAL;
    *bytes = 256 + (size_t)batch * sizeof(float);
    return CPB_OK;
}

int cpb_viterbi_decode_punctured(const cpbTrellis *t, const float *llr_punct_dev, int64_t batch, int64_t n_kept,
                                 const int32_t *punct_vec_host, int punct_len, int64_t n_depunct, int tb_depth, int mode,
                                 uint8_t *out_bits_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    if (mode != CPB_VITERBI_SOFT && mode != CPB_VITERBI_UNQUANTIZED) return CPB_EINVAL;
    if (t && batch == 0) return CPB_OK;
    if (!t || !llr_punct_dev || !out_bits_dev || !punct_vec_host || batch < 0 || n_kept < 0 || n_depunct <= 0) return CPB_EINVAL;
    if (punct_len < 1 || punct_len > 32) return CPB_EUNSUPPORTED;
    uint32_t mask = 0;
    int ones = 0;
    for (int i = 0; i < punct_len; ++i)
        if (punct_vec_host[i] == 1) { mask |= 1u << i; ++ones; }
    // values the depuncturing consumes (convcode.py:796-799 indexes the punctured array: IndexError when it is too short)
    const int64_t need = (n_depunct / punct_len) * ones + __builtin_popcount(mask & ((1u << (n_depunct % punct_len)) - 1u));
    if (need > n_kept) return CPB_EINVAL;
    int64_t L, T;
    cpb_viterbi_sizes(t, n_depunct, &L, &T);
    const int D = resolve_depth(t, L, tb_depth);
    if (L <= 0 || D < 2 || T < D - 1 || T > (1 << 24)) return CPB_EINVAL;
    if (!use_fast(t, D, mode, CPB_F32)) return CPB_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    fast::Params p{};
    int rc = fast_params(p, llr_punct_dev, n_depunct, batch, L, T, D, mode, out_bits_dev);
    if (rc) return rc;
    p.punct_mask = mask; p.punct_len = punct_len; p.n_kept = n_kept;
    Scratch ws;
    rc = ws.acquire(workspace_dev, workspace_bytes, 256 + (size_t)batch * sizeof(float), st);
    if (rc) return rc;
    // the erasures are zeros: the frame's scale is the largest magnitude among the values the depuncturing uses
    rc = frame_scales(p, llr_punct_dev, n_kept, need, ws.ptr, st);
    if (!rc) rc = launch_fast<1, 2>(t, p, st);
    ws.release();
    return rc;
}

}  // extern "C"
