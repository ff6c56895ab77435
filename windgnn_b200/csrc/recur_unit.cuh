// GRU recurrence, throughput kernel (second generation): gate values never leave registers.
//
// Reference: `gru_out, _ = self.gru(hidden2)` at src/step6_gcn_gru_combined_model.py:23 (module
// built at :11), PyTorch gate convention (rows r, z, n) — see recur.cuh for the equations.
//
// gru_recur_kernel (recur.cuh) tiles the per-step product h . W_hh^T by gate COLUMNS, so the r, z
// and n values of one hidden unit end up in different threads and have to meet in shared memory
// (merge phase, a barrier, a separate gate phase); its two 16-sequence groups hand the FMA pipe to
// each other, which leaves one GEMM warp per scheduler and the pipe half idle (ncu r01: 57.6 %).
//
// Here a thread owns the r, z and n columns of TWO hidden units (2p, 2p+1) for the R sequences of
// its group:   acc[i][g] (float2 over the unit pair)  +=  h[i][k] * (W_g[k][2p], W_g[k][2p+1])
// — FFMA2 with h as the broadcast scalar.  When the product is done the thread already holds
// everything a GRU cell needs for its R x 2 (sequence, unit) items: gi of the step sits in a per-group
// shared-memory tile (one bulk async copy per sequence row, issued one step ahead by one thread and
// completing on the group's mbarrier), the previous state of those items lives in registers.  No merge phase, no gh round trip; the only
// exchange per step is the new state, written to the other half of a double-buffered h tile,
// followed by ONE named barrier among the group's warps.
//
// A CTA (8 warps) holds W_hh^T once (127 KB at H = 102) and runs 8 / WPG independent groups of R
// sequences (WPG = warps per group = ceil(H / 64)); the groups drift apart, so one group's gate
// phase (MUFU) overlaps another's product (FMA) on the same scheduler.  R is chosen per launch
// (4 .. 8) so that the grid is one full wave: 4096 sequences -> 147 CTAs of 4 x 7.
//
// Every output's sum runs over k ascending in one FMA chain and the gate expressions are those of
// gru_recur_regw_kernel (recur.cuh), which takes the small batches of the shipped models: the two
// kernels are bit-identical (tested), so the kernel choice — which depends on the batch size — never
// changes a result.
#pragma once

#include "recur.cuh"
#include "wg_common.cuh"

namespace wg {

constexpr int kRuWarps = 8;
constexpr int kRuThreads = kRuWarps * 32;
constexpr int kRuMaxR = 8;
constexpr int kRuMinR = 4;

__host__ __device__ inline int recur_u_hp2(int H) { return round_up(H, 2); }
// warps per group: a lane owns one unit pair
__host__ __device__ inline int recur_u_wpg(int H) { return recur_u_hp2(H) / 2 <= 32 ? 1 : 2; }
__host__ __device__ inline bool recur_u_applies(int H) { return recur_u_hp2(H) / 2 <= 64; }
// gi tiles in flight per group.  One-warp groups (H <= 64) have a product of a few hundred cycles per step — shorter
// than the latency of the bulk copy that brings the next step's gi — so their tile is a ring filled kRuGiRing steps
// ahead; two-warp groups (9 K cycles of product per step, shared memory full of W_hh) keep one tile.
constexpr int kRuGiRing = 4;
__host__ __device__ inline int recur_u_nb(int H) { return recur_u_wpg(H) == 1 ? kRuGiRing : 1; }
// h rows: KP floats, padded so that consecutive rows start in different 16-byte bank groups
__host__ __device__ inline int recur_u_hs_stride(int KP) { return ((KP / 4) & 1) ? KP : KP + 4; }
__host__ __device__ inline size_t recur_u_smem_floats(int H, int R) {
    const int KP = round_up(H, 4), HP2 = recur_u_hp2(H), WPG = recur_u_wpg(H), NGRP = kRuWarps / WPG;
    const int GP = round_up(3 * H, 8);
    size_t n = (size_t)KP * 3 * HP2;                          // W_hh^T as [k][gate][unit]
    n = round_up((int)n, 4);
    n += 2 * (size_t)NGRP * R * recur_u_hs_stride(KP);        // h, double buffered
    n += (size_t)recur_u_nb(H) * NGRP * R * GP;               // gi tiles (ring of recur_u_nb steps), per group
    n += (size_t)round_up(HP2, 4);                            // b_hn
    n += 2 * (size_t)NGRP * recur_u_nb(H);                    // one mbarrier per group and ring slot
    return n;
}

#ifdef WG_RC_TRACE
// debug build only: clock stamps of CTA 0, per warp and step (5 stamps per step)
__device__ long long g_ru_trace[8 * 256 * 5];
#define WG_RU_TRACE(slot)                                                                                   \
    do {                                                                                                    \
        if (blockIdx.x == 0 && (tid & 31) == 0 && t < 256) g_ru_trace[((tid >> 5) * 256 + t) * 5 + (slot)] = clock64(); \
    } while (0)
#else
#define WG_RU_TRACE(slot) do { } while (0)
#endif

template <int R>
struct RuFrag {
    float4 h[R];      // h[i] = hs[row i][k .. k+3]
    float2 w[4][3];   // w[kk][g] = W_g[k + kk][2p .. 2p+1]
};

// GI  [B*T][ldg]   gi with b_ih (+ b_hh for r, z) folded in, column g*H + j; ldg = 3H rounded up to 8
// Whu [KP][3][HP2] W_hh^T, Whu[k][g][j] = w_hh[g*H + j][k], zero padded
// out [B][T][H];   gsave (SAVE): [B*T][ldsave] = [r | z | n | W_hn h + b_hn]
// HT > 0: the hidden size is the compile-time constant HT (every shared-memory offset becomes an
// immediate); HT == 0: H is the runtime argument.
// WIN: a WinMode (recur.cuh).  kWinLast and kWinAll read sequence b's gi rows from GI + row0[b] * ldg (windows over one
// table's gi rows); kWinLast stores only h at t = T-1, to out [B][H].  The product and the gate math are unchanged.
template <int R, int WPG, bool SAVE, int HT, int WIN = kWinOff>
__global__ void __launch_bounds__(kRuThreads, 1)
    gru_recur_unit_kernel(const float* __restrict__ GI, const float* __restrict__ Whu, const float* __restrict__ bhn,
                          float* __restrict__ out, long long B, int T, int H_rt,
                          float* __restrict__ gsave, int ldsave, int handover,
                          const long long* __restrict__ row0) {
    constexpr bool ROW0 = WIN != kWinOff, LAST = WIN == kWinLast;
    constexpr int NGRP = kRuWarps / WPG;   // groups per CTA
    constexpr int NG = WPG * 32;           // threads per group
    constexpr int NB = WPG == 1 ? kRuGiRing : 1;   // gi ring slots per group (recur_u_nb)
    // Hand-over of the FMA pipe (handover != 0; one-warp groups only).  Warp w issues on scheduler w % 4, so the
    // one-warp groups g and g + NGRP/2 share a scheduler.  With the hand-over the second group starts its product
    // when the first has finished its own, so one group's gate phase (MUFU, stores) runs under the other's
    // product: barrier X = "first group's product done", Y = "second group's product done" (arrive = signal,
    // sync = wait).  Measured: H = 21 0.395 -> 0.358 ms at 4096 sequences.
    constexpr int HALF = NGRP / 2;
    constexpr int kBarBase = WPG == 1 ? 1 : 1 + NGRP;   // WPG == 1: the group barrier is a __syncwarp
    extern __shared__ __align__(16) float smem[];
    const int H = HT > 0 ? HT : H_rt;
    const int KP = round_up(H, 4), HP2 = recur_u_hp2(H), NS = HP2 >> 1, ldg = round_up(3 * H, 8);
    const int RS = recur_u_hs_stride(KP);
    float* Ws = smem;                                                // [KP][3][HP2]
    float* hs = Ws + round_up(KP * 3 * HP2, 4);                      // [2][NGRP * R][RS]
    float* gis = hs + 2 * NGRP * R * RS;                             // [NB][NGRP][R][ldg]
    float* bns = gis + NB * NGRP * R * ldg;                          // [HP2]
    uint64_t* gbar = reinterpret_cast<uint64_t*>(bns + round_up(HP2, 4));   // [NGRP][NB]

    const int tid = threadIdx.x;
    // warp w issues on scheduler w % 4.  Two-warp groups take warps g and g + 4: BOTH warps of a group then sit on
    // one scheduler, which they have to themselves — they run the product together (two warps saturate the FMA
    // pipe, one does not: 2.2 vs 3 cycles per FFMA2) and reach the group barrier together.  (Warps 2g, 2g + 1:
    // each warp shares its scheduler with another group's warp; the skew cost 1.1 K cycles of barrier wait per step.)
    const int grp = WPG == 2 ? ((tid >> 5) & (NGRP - 1)) : tid / NG;
    const int p = WPG == 2 ? ((tid >> 5) / NGRP) * 32 + (tid & 31) : tid - grp * NG;   // unit pair of this thread
    const bool second = grp >= HALF;
    const int bar_x = kBarBase + 2 * (grp - (second ? HALF : 0)), bar_y = bar_x + 1;
    const bool active = p < NS;
    const int pc = active ? p : NS - 1;    // clamped: idle lanes load valid addresses and store nothing
    const int j0 = 2 * pc;
    const bool has1 = j0 + 1 < H;          // the pair's second unit exists (H odd: not in the last slot)
    const long long b0 = (long long)blockIdx.x * (NGRP * R) + grp * R;   // first sequence of the group
    const int H2 = 2 * H;
    const long long left = B - b0;
    const int nvalid = left >= R ? R : (left > 0 ? (int)left : 0);       // sequences of this group that exist

    {
        const int n4 = KP * 3 * HP2 / 4;   // KP % 4 == 0
        const float4* src = reinterpret_cast<const float4*>(Whu);
        float4* dst = reinterpret_cast<float4*>(Ws);
        for (int e = tid; e < n4; e += kRuThreads) dst[e] = __ldg(src + e);
    }
    for (int e = tid; e < 2 * NGRP * R * RS; e += kRuThreads) hs[e] = 0.0f;
    for (int e = tid; e < NB * NGRP * R * ldg; e += kRuThreads) gis[e] = 0.0f;
    for (int e = tid; e < HP2; e += kRuThreads) bns[e] = e < H ? __ldg(bhn + e) : 0.0f;
    if (tid < NGRP * NB) mbar_init(&gbar[tid], 1);
    if (tid == 0) fence_mbar_init();

    // gi(t) of the group's sequences: one bulk async copy per row (ldg * 4 bytes, 16-byte multiple) into slot
    // t % NB of the group's tile ring, completion counted on that slot's mbarrier.  Issued by one thread AFTER the
    // group barrier that ends step t - NB, i.e. when every thread of the group has read gi(t - NB).
    float* gi_ring = gis + grp * R * ldg;        // slot stride: NGRP * R * ldg
    uint64_t* gi_bar = gbar + grp * NB;
    const float* gwin[ROW0 ? R : 1];             // ROW0: gi row 0 of each of the group's sequences
    if (ROW0 && p == 0) {
#pragma unroll
        for (int i = 0; i < (ROW0 ? R : 1); ++i) gwin[i] = GI + (size_t)(i < nvalid ? row0[b0 + i] : 0) * ldg;
    }
    auto fetch_gi = [&](int t) {
        if (nvalid > 0) {
            const int slot = NB == 1 ? 0 : t % NB;
            float* tile = gi_ring + slot * (NGRP * R * ldg);
            mbar_expect_tx(&gi_bar[slot], (unsigned)(nvalid * ldg * 4));
            if (ROW0) {
#pragma unroll
                for (int i = 0; i < (ROW0 ? R : 1); ++i)
                    if (i < nvalid)
                        bulk_g2s(tile + i * ldg, gwin[i] + (size_t)t * ldg, (unsigned)(ldg * 4), &gi_bar[slot]);
            } else {
                for (int i = 0; i < nvalid; ++i)
                    bulk_g2s(tile + i * ldg, GI + ((size_t)(b0 + i) * T + t) * ldg, (unsigned)(ldg * 4),
                             &gi_bar[slot]);
            }
        }
    };

    __syncthreads();   // zero fills and barrier inits are done before any async copy may land
    if (p == 0)
        for (int t = 0; t < NB && t < T; ++t) fetch_gi(t);

    float2 hprev[R];   // h_{t-1} of this thread's items
#pragma unroll
    for (int i = 0; i < R; ++i) hprev[i] = make_float2(0.0f, 0.0f);
    const float2 bn = make_float2(bns[j0], has1 ? bns[j0 + 1] : 0.0f);
    const float* wbase = Ws + j0;
    const bool out_vec = (reinterpret_cast<uintptr_t>(out) & 7) == 0 && (H & 1) == 0;
    const bool save_vec = SAVE && (reinterpret_cast<uintptr_t>(gsave) & 7) == 0 && (ldsave & 1) == 0 && (H & 1) == 0;
    const bool gi_vec = (H & 1) == 0;      // g*H + j0 even: 8-byte reads of the gi tile
    // running output pointers: + H per step (LAST: one row per sequence, written at the last step)
    float* op0 = out + (size_t)b0 * (LAST ? 1 : T) * H + j0;
    const size_t o_seq = (size_t)(LAST ? 1 : T) * H;
    float* gs0 = SAVE ? gsave + (size_t)b0 * T * ldsave + j0 : nullptr;
    const size_t s_seq = (size_t)T * ldsave;

    for (int t = 0; t < T; ++t) {
        const float* hcur = hs + ((t & 1) * NGRP + grp) * R * RS;           // h_{t-1}: read
        float* hnxt = hs + (((t + 1) & 1) * NGRP + grp) * R * RS;           // h_t: written
        if (handover) {
            if (second) group_barrier(bar_x, 2 * NG);
            else if (t > 0) group_barrier(bar_y, 2 * NG);
        }
        WG_RU_TRACE(0);
        // ================= product: acc[i][g] = sum_k h[i][k] * W_g[k][2p, 2p+1] =================
        float2 acc[R][3];
#pragma unroll
        for (int i = 0; i < R; ++i)
#pragma unroll
            for (int g = 0; g < 3; ++g) acc[i][g] = make_float2(0.0f, 0.0f);
        if (t > 0) {   // h_{-1} = 0: the product is zero at t == 0
            const float* hp = hcur;
            const float* wp = wbase;
            const int wk = 3 * HP2;   // floats per k
            auto load_frag = [&](RuFrag<R>& f) {
#pragma unroll
                for (int i = 0; i < R; ++i) f.h[i] = *reinterpret_cast<const float4*>(hp + i * RS);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
#pragma unroll
                    for (int g = 0; g < 3; ++g)
                        f.w[kk][g] = *reinterpret_cast<const float2*>(wp + kk * wk + g * HP2);
                hp += 4;
                wp += 4 * wk;
            };
            auto mma_frag = [&](const RuFrag<R>& f) {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
                    for (int i = 0; i < R; ++i) {
                        const float hv = kk == 0 ? f.h[i].x : kk == 1 ? f.h[i].y : kk == 2 ? f.h[i].z : f.h[i].w;
                        const float2 hh = make_float2(hv, hv);   // FFMA2 broadcasts a scalar operand
#pragma unroll
                        for (int g = 0; g < 3; ++g) acc[i][g] = __ffma2_rn(hh, f.w[kk][g], acc[i][g]);
                    }
                }
            };
            // software pipeline over KP / 4 fragments, two register buffers
            RuFrag<R> fa, fb;
            load_frag(fa);
            int k4 = 4;
#pragma unroll 1
            for (; k4 + 4 < KP; k4 += 8) {
                load_frag(fb);
                mma_frag(fa);
                load_frag(fa);
                mma_frag(fb);
            }
            if (k4 < KP) {   // even number of fragments: one more pair
                load_frag(fb);
                mma_frag(fa);
                mma_frag(fb);
            } else {
                mma_frag(fa);
            }
        }
        if (handover) {
            if (!second) group_arrive(bar_x, 2 * NG);
            else if (t + 1 < T) group_arrive(bar_y, 2 * NG);
        }
        WG_RU_TRACE(1);
        // ================= gates, straight from the accumulators =================
        const int slot = NB == 1 ? 0 : t % NB;
        const float* gi_tile = gi_ring + slot * (NGRP * R * ldg);
        if (nvalid > 0) mbar_wait(&gi_bar[slot], (unsigned)((t / NB) & 1));   // gi(t) has landed
        float2 gi[3][R];
#pragma unroll
        for (int g = 0; g < 3; ++g)
#pragma unroll
            for (int i = 0; i < R; ++i) {
                const float* gp = gi_tile + i * ldg + g * H + j0;
                if (gi_vec) {
                    gi[g][i] = *reinterpret_cast<const float2*>(gp);
                } else {
                    gi[g][i].x = gp[0];
                    gi[g][i].y = has1 ? gp[1] : 0.0f;
                }
            }
        WG_RU_TRACE(2);
#pragma unroll
        for (int i = 0; i < R; ++i) {
            float2 hn, r, z, n, hnew;
            // the same expressions, in the same order, as the merge + gate phases of gru_recur_kernel
            r.x = sigmoid_f(gi[0][i].x + acc[i][0].x);
            r.y = sigmoid_f(gi[0][i].y + acc[i][0].y);
            z.x = sigmoid_f(gi[1][i].x + acc[i][1].x);
            z.y = sigmoid_f(gi[1][i].y + acc[i][1].y);
            hn.x = acc[i][2].x + bn.x;
            hn.y = acc[i][2].y + bn.y;
            n.x = tanh_f(gi[2][i].x + r.x * hn.x);
            n.y = tanh_f(gi[2][i].y + r.y * hn.y);
            hnew.x = (hprev[i].x - n.x) * z.x + n.x;
            hnew.y = has1 ? (hprev[i].y - n.y) * z.y + n.y : 0.0f;
            hprev[i] = hnew;
            if (active) {
                *reinterpret_cast<float2*>(hnxt + i * RS + j0) = hnew;
                if (i < nvalid && (!LAST || t == T - 1)) {
                    float* op = op0 + i * o_seq;
                    if (out_vec) {
                        *reinterpret_cast<float2*>(op) = hnew;
                    } else {
                        op[0] = hnew.x;
                        if (has1) op[1] = hnew.y;
                    }
                    if (SAVE) {
                        float* gs = gs0 + i * s_seq;
                        if (save_vec) {
                            *reinterpret_cast<float2*>(gs) = r;
                            *reinterpret_cast<float2*>(gs + H) = z;
                            *reinterpret_cast<float2*>(gs + H2) = n;
                            *reinterpret_cast<float2*>(gs + H2 + H) = hn;
                        } else {
                            gs[0] = r.x; gs[H] = z.x; gs[H2] = n.x; gs[H2 + H] = hn.x;
                            if (has1) { gs[1] = r.y; gs[H + 1] = z.y; gs[H2 + 1] = n.y; gs[H2 + H + 1] = hn.y; }
                        }
                    }
                }
            }
        }
        if (!LAST) op0 += H;
        if (SAVE) gs0 += ldsave;
        // h_t complete for the group before anyone reads it; the buffer written at step t+1 is the one
        // read at step t, which every warp of the group has finished with once it arrives here.  The same
        // barrier tells the fetching thread that everyone has read gi(t).
        WG_RU_TRACE(3);
        if (WPG == 1) __syncwarp();
        else group_barrier(1 + grp, NG);
        if (p == 0 && t + NB < T) fetch_gi(t + NB);   // refills the slot just read; lands during the next product(s)
        WG_RU_TRACE(4);
    }
}

}  // namespace wg
