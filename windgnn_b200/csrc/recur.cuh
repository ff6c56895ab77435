// GRU recurrence — the serial part of nn.GRU (h0 = 0), all T steps inside ONE launch.
//
// Reference: `gru_out, _ = self.gru(hidden2)` at src/step6_gcn_gru_combined_model.py:23 (module
// built at :11), PyTorch gate convention (rows r, z, n):
//     gh = W_hh h + b_hh
//     r = sigma(gi_r + gh_r)   z = sigma(gi_z + gh_z)   n = tanh(gi_n + r * gh_n)
//     h' = (h - n) * z + n
// gi (with b_ih, and b_hh for r and z, already added) comes from the input-projection kernel.
//
// gru_recur_kernel serves the hidden sizes that gru_recur_unit_kernel (recur_unit.cuh) cannot fit in
// shared memory, H = 125 .. 360.  A CTA owns 32 sequences for all T steps.  W_hh^T ([k][n], zero
// padded to KP x NP; too large for shared memory at these sizes) is read through L1 / L2 every step,
// the hidden state of the 32 sequences lives in shared memory; nothing but gi (read) and h
// (written) touches HBM inside the time loop.  The 16 warps form TWO independent groups of 16
// sequences that only ever synchronise among themselves (named barriers), so one group's gate phase
// (MUFU-bound) overlaps the other group's GEMM (FMA-bound).  Per step:
//   GEMM  : acc[b][n] = sum_k h[b][k] * W[k][n] on the FMA pipe with packed FFMA2 (sm_100a):
//           acc2[b][(n, n+1)] += h[b][k] (scalar operand, broadcast) * (W[k][n], W[k][n+1]).
//           A warp covers 16 sequences x 80 gate columns, a thread 4 x 10 (five column pairs);
//           operand fragments of four k's are double-buffered in registers so the LDS latency
//           hides behind the previous fragment's 80 FFMA2.
//   merge : each thread adds its accumulators onto the gi chunks that IT prefetched with
//           cp.async during the GEMM (no barrier needed: a thread only waits for its own
//           copies); the n-gate part of gh is kept apart because r multiplies it.
//   gates : one (sequence, hidden unit) item per thread-slot, lanes along the hidden index so
//           the h stores to HBM are coalesced.
#pragma once

#include "wg_common.cuh"

namespace wg {

constexpr int kRcBT = 32;    // sequences per CTA (two groups of 16)
constexpr int kRcCB = 80;    // gate columns per warp
constexpr int kRcWarps = 16;   // eight per group; a warp loops over every eighth 80-column block

__host__ __device__ inline int recur_np(int G) { return round_up(G, kRcCB); }
// hidden-state rows: KP floats padded so that four consecutive rows start in distinct bank groups
__host__ __device__ inline int recur_hs_stride(int KP) { return ((KP / 4) & 1) ? KP : KP + 4; }
// timesteps staged in shared memory per bulk store of h: the smallest count that makes one
// sequence's staged block (TS * H floats) a multiple of 16 bytes
__host__ __device__ inline int recur_stage_steps(int H) { return (H % 4 == 0) ? 1 : (H % 2 == 0) ? 2 : 4; }
__host__ __device__ inline size_t recur_smem_floats(int KP, int GP, int H = 0, int TS = 0) {
    size_t n = (size_t)round_up(kRcBT * TS * H, 4);  // staging of h for the bulk stores (TS = 0: none)
    n += (size_t)kRcBT * recur_hs_stride(KP);  // hs
    n += (size_t)kRcBT * GP;                   // gi tile (r,z columns become gi + gh)
    n += (size_t)kRcBT * KP;                   // gh of the n gate
    n += (size_t)KP;                           // b_hn
    return n;
}

__device__ __forceinline__ void group_barrier(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void group_arrive(int id, int nthreads) {
    asm volatile("bar.arrive %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}

// one operand fragment: four k's of this thread's 4 rows and 10 columns
struct RcFrag {
    float4 h[4];      // h[i] = hs[row i][k .. k+3]
    float4 wa[4];     // W[k + kk][cA .. cA+3]
    float4 wb[4];     // W[k + kk][cB .. cB+3]
    float2 wc[4];     // W[k + kk][cC .. cC+1]
};

// WIN: windows over one table's gi rows (see gru_recur_unit_kernel): row rbase + 4i of the CTA reads its gi from
// GI + row0[b] * ldg, and only h at t = T-1 is stored, directly to out [B][H] (the launch passes TS = 0: no staging)
template <bool WIN = false>
__global__ void __launch_bounds__(kRcWarps * 32, 1)
    gru_recur_kernel(const float* __restrict__ GI, const float* __restrict__ WhT,
                     const float* __restrict__ bhn, float* __restrict__ out, long long B, int T, int H,
                     int ldg, int KP, int NP, int TS, const long long* __restrict__ row0) {
    constexpr int NT = kRcWarps * 32;
    constexpr int WG = kRcWarps / 2;   // warps per group
    constexpr int NG = WG * 32;      // threads per group
    constexpr int GB = kRcBT / 2;    // sequences per group
    extern __shared__ __align__(16) float smem[];
    const int RS = recur_hs_stride(KP);
    float* hs = smem;
    float* gis = hs + kRcBT * RS;          // [32][ldg]
    float* ghn = gis + kRcBT * ldg;        // [32][KP]
    float* bns = ghn + kRcBT * KP;         // [KP]
    float* stage = bns + KP;               // [32][TS][H] h of the last TS steps (TS > 0)
    // bulk (TMA) stores of h need 16-byte aligned, 16-byte-multiple spans per sequence
    const bool bulk_ok = TS > 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (((long long)T * H) & 3) == 0 &&
                         ((TS * H) & 3) == 0;

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int grp = warp / WG;             // 0 or 1: which 16 sequences
    const int gwarp = warp - grp * WG;     // warp index inside the group
    const int gtid = tid - grp * NG;
    const long long b0 = (long long)blockIdx.x * kRcBT;
    const int H2 = 2 * H;

    for (int e = tid; e < kRcBT * RS; e += NT) hs[e] = 0.0f;
    for (int e = tid; e < kRcBT * ldg; e += NT) gis[e] = 0.0f;
    for (int e = tid; e < kRcBT * KP; e += NT) ghn[e] = 0.0f;
    for (int e = tid; e < KP; e += NT) bns[e] = e < H ? __ldg(bhn + e) : 0.0f;

    // ---- GEMM-phase coordinates ----
    const int ln = lane & 7;   // column slot within the warp's 80 columns
    const int bg = lane >> 3;  // row group
    const int n_cb = NP / kRcCB;           // 80-column blocks; this warp takes gwarp, gwarp + WG, ...
    const int rbase = grp * GB + bg;       // rows rbase + 4 i

    // WIN: gi row 0 of this thread's rows rbase + 4i
    const float* gwin[WIN ? 4 : 1];
    if (WIN) {
#pragma unroll
        for (int i = 0; i < (WIN ? 4 : 1); ++i) {
            const long long b = b0 + rbase + 4 * i;
            gwin[i] = GI + (size_t)(b < B ? row0[b] : 0) * ldg;
        }
    }
    // this thread's chunks of the gi tile of step t: per row 16 + 16 + 8 bytes per column block
    auto prefetch_gi = [&](int t) {
        for (int cb = gwarp; cb < n_cb; cb += WG) {
            const int cA = cb * kRcCB + ln * 4, cB = cA + 32, cC = cb * kRcCB + 64 + ln * 2;
            const float* src = GI + ((size_t)(b0 + rbase) * T + t) * ldg;   // row rbase; rows are 4*T*ldg apart
            float* dst = gis + rbase * ldg;
            const size_t src_step = (size_t)4 * T * ldg;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (WIN) src = gwin[WIN ? i : 0] + (size_t)t * ldg;
                if (b0 + rbase + 4 * i < B) {
                    if (cA < ldg) cp_async16(dst + cA, src + cA, true);
                    if (cB < ldg) cp_async16(dst + cB, src + cB, true);
                    if (cC < ldg) cp_async8(dst + cC, src + cC);
                }
                src += src_step;
                dst += 4 * ldg;
            }
        }
        cp_async_commit();
    };

    __syncthreads();   // zero fills are done before any async copy may land
    prefetch_gi(0);

    const float* hrow = hs + rbase * RS;
    const int h_step = 4 * RS;
    for (int t = 0; t < T; ++t) {
        // The two groups take turns on the FMA pipe: group 0 runs GEMM(t) while group 1 does the
        // merge / gates of step t-1, then they swap.  Barrier 3: "group 0 finished its GEMM",
        // barrier 4: "group 1 finished its GEMM" (arrive = signal, sync = wait; NT participants).
        if (grp == 0) {
            if (t > 0) group_barrier(4, NT);
        } else {
            group_barrier(3, NT);
        }
        // ================= GEMM + merge =================
        bool handed_over = false;
        for (int cb = gwarp; cb < n_cb; cb += WG) {
            const int cA = cb * kRcCB + ln * 4, cB = cA + 32, cC = cb * kRcCB + 64 + ln * 2;
            float2 acc[4][5];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int p = 0; p < 5; ++p) acc[i][p] = make_float2(0.0f, 0.0f);

            const float* hp = hrow;            // + 4 floats per fragment
            const float* wp = WhT + cA;        // + 4 * NP floats per fragment
            auto load_frag = [&](RcFrag& f) {
#pragma unroll
                for (int i = 0; i < 4; ++i) f.h[i] = *reinterpret_cast<const float4*>(hp + i * h_step);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const float* w = wp + kk * NP;
                    f.wa[kk] = __ldg(reinterpret_cast<const float4*>(w));
                    f.wb[kk] = __ldg(reinterpret_cast<const float4*>(w + 32));
                    f.wc[kk] = __ldg(reinterpret_cast<const float2*>(w + 64 - 2 * ln));
                }
                hp += 4;
                wp += 4 * NP;
            };
            auto mma_frag = [&](const RcFrag& f) {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float hv = kk == 0 ? f.h[i].x : kk == 1 ? f.h[i].y : kk == 2 ? f.h[i].z : f.h[i].w;
                        const float2 hh = make_float2(hv, hv);  // FFMA2 broadcasts a scalar operand
                        acc[i][0] = __ffma2_rn(hh, make_float2(f.wa[kk].x, f.wa[kk].y), acc[i][0]);
                        acc[i][1] = __ffma2_rn(hh, make_float2(f.wa[kk].z, f.wa[kk].w), acc[i][1]);
                        acc[i][2] = __ffma2_rn(hh, make_float2(f.wb[kk].x, f.wb[kk].y), acc[i][2]);
                        acc[i][3] = __ffma2_rn(hh, make_float2(f.wb[kk].z, f.wb[kk].w), acc[i][3]);
                        acc[i][4] = __ffma2_rn(hh, f.wc[kk], acc[i][4]);
                    }
                }
            };
            if (t > 0) {  // h_{-1} = 0: the product is zero at t == 0
                // software pipeline over KP / 4 fragments; branch-free body so the fragment
                // registers are written by the loads themselves
                RcFrag fa, fb;
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
            if (cb + WG >= n_cb) {  // last column block of this warp: hand the FMA pipe over
                if (grp == 0) group_arrive(3, NT);
                else if (t + 1 < T) group_arrive(4, NT);
                handed_over = true;
            }
            cp_async_wait<0>();  // this thread's chunks of gi(t) have landed
            // merge: r/z columns accumulate onto gi (vector read-modify-write), n-gate columns go to
            // ghn; a chunk that straddles a gate boundary (or the padding) takes the element path.
            // The class of a chunk is the same for the thread's four rows.
            auto merge_chunk = [&](int n0, auto width, int p0) {
                constexpr int W = decltype(width)::value;
                if (n0 + W <= H2) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        float* g = gis + (rbase + 4 * i) * ldg + n0;
                        if (W == 4) {
                            float4 v = *reinterpret_cast<float4*>(g);
                            v.x += acc[i][p0].x; v.y += acc[i][p0].y; v.z += acc[i][p0 + 1].x; v.w += acc[i][p0 + 1].y;
                            *reinterpret_cast<float4*>(g) = v;
                        } else {
                            float2 v = *reinterpret_cast<float2*>(g);
                            v.x += acc[i][p0].x; v.y += acc[i][p0].y;
                            *reinterpret_cast<float2*>(g) = v;
                        }
                    }
                } else if (n0 < 3 * H) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        float* g = gis + (rbase + 4 * i) * ldg;
                        float* gn = ghn + (rbase + 4 * i) * KP;
#pragma unroll
                        for (int c = 0; c < W; ++c) {
                            const int n = n0 + c;
                            const float a = (c & 1) ? acc[i][p0 + (c >> 1)].y : acc[i][p0 + (c >> 1)].x;
                            if (n < H2) g[n] += a;
                            else if (n < 3 * H) gn[n - H2] = a;
                        }
                    }
                }
            };
            merge_chunk(cA, IntC<4>{}, 0);
            merge_chunk(cB, IntC<4>{}, 2);
            merge_chunk(cC, IntC<2>{}, 4);
        }
        if (!handed_over) {  // a warp without a column block still takes part in the hand-over
            if (grp == 0) group_arrive(3, NT);
            else if (t + 1 < T) group_arrive(4, NT);
        }
        if (bulk_ok && gtid < GB) bulk_wait_read();  // the previous bulk store has read its staging rows
        group_barrier(1 + grp, NG);

        // ================= gate phase =================
        // A thread owns hidden unit(s) j and walks the group's 16 sequences: every address is a
        // running pointer (no index arithmetic), lanes lie along j (conflict-free shared accesses),
        // and four sequences are in flight at once so their MUFU chains overlap.
        for (int j = gtid; j < H; j += NG) {
            const float bn = bns[j];
            // distinct buffers: __restrict__ lets the loads of later sequences pass earlier stores
            const float* __restrict__ g = gis + (grp * GB) * ldg + j;
            const float* __restrict__ gn = ghn + (grp * GB) * KP + j;
            float* __restrict__ hp = hs + (grp * GB) * RS + j;
            float* __restrict__ sp = stage + (grp * GB) * TS * H + (TS > 0 ? (t % TS) * H : 0) + j;
            float* __restrict__ op = out + ((size_t)(b0 + grp * GB) * (WIN ? 1 : T) + (WIN ? 0 : t)) * H + j;
            const size_t o_step = (size_t)(WIN ? 1 : T) * H;
            const int s_step = TS * H;
            // pass 1: all 16 new states into registers (no store in between, so the loads and MUFU
            // chains of different sequences overlap); pass 2: the stores
            float hnew[GB];
#pragma unroll
            for (int bl = 0; bl < GB; ++bl) {
                const float r = sigmoid_f(g[bl * ldg]);
                const float z = sigmoid_f(g[bl * ldg + H]);
                const float hn = gn[bl * KP] + bn;
                const float n = tanh_f(g[bl * ldg + H2] + r * hn);
                hnew[bl] = (hp[bl * RS] - n) * z + n;
            }
#pragma unroll
            for (int bl = 0; bl < GB; ++bl) {
                hp[bl * RS] = hnew[bl];
                if (TS > 0) sp[bl * s_step] = hnew[bl];
                else if ((!WIN || t == T - 1) && b0 + grp * GB + bl < B) op[bl * o_step] = hnew[bl];
            }
        }
        if (TS > 0) asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // staged h -> async proxy
        group_barrier(1 + grp, NG);
        if (TS > 0 && ((t % TS) == TS - 1 || t == T - 1)) {
            // flush the staged steps t0 .. t of this group's 16 sequences to out[b][t0 .. t][:]
            const int t0 = t - (t % TS), nst = t - t0 + 1;
            if (bulk_ok && nst == TS) {
                if (gtid < GB) {
                    const int b = grp * GB + gtid;
                    if (b0 + b < B) {
                        bulk_s2g(out + ((size_t)(b0 + b) * T + t0) * H, stage + b * TS * H, (unsigned)(TS * H * 4));
                        bulk_commit();
                    }
                }
            } else {
                const int per_seq = nst * H;
                for (int e = gtid; e < GB * per_seq; e += NG) {
                    const int bl = e / per_seq, r = e - bl * per_seq;
                    const int b = grp * GB + bl;
                    if (b0 + b < B) out[((size_t)(b0 + b) * T + t0) * H + r] = stage[b * TS * H + r];
                }
                group_barrier(1 + grp, NG);  // the staging rows are free again
            }
        }
        if (t + 1 < T) prefetch_gi(t + 1);  // lands during the next GEMM
    }
    if (bulk_ok && gtid < GB) bulk_wait_read();  // shared memory must outlive the last bulk store's reads
}

// ---------------------------------------------------------------------------------------------
// Small-batch recurrence: 4 sequences per CTA, W_hh IN REGISTERS (compile-time contraction length KPT).
//
// The throughput kernels spend a fixed time per timestep whatever the batch; a few sequences — the
// reference's own call pattern (`model(adj_matrix, batch_x)` with batch 1, src/main.py:66,102) or a
// small per-GPU shard — leave most of the machine idle.  For the contraction lengths of the shipped
// models (KP = 24: the 7-station model, KP = 104: the 34-station model) this kernel runs instead
// when the batch is small.  A thread owns one gate COLUMN and keeps its KPT weights in registers for
// the whole kernel (streaming W_hh^T — 127 KB at H = 102 — out of shared memory cost ~1000 cycles of
// LSU time per step even for ONE sequence); a step's product is KPT FFMAs per sequence in one
// dependent chain (k ascending: bit-identical to every other recurrence kernel), fed by broadcast
// 16-byte loads of h.  Shared memory holds only h, gi (double buffered, prefetched with cp.async one
// step ahead) and gh (17 KB).  Serves 3H (padded) <= 320.
// ---------------------------------------------------------------------------------------------
constexpr int kRsBT = 4;          // sequences per CTA
constexpr int kRwThreads = 320;   // 10 warps >= the 306 gate columns of H = 102

__host__ __device__ inline size_t recur_regw_smem_floats(int KP, int NP, int GP) {
    return (size_t)kRsBT * (KP + 4) + 2 * (size_t)kRsBT * GP + (size_t)kRsBT * NP + (size_t)KP;
}

// WIN: windows over one table's gi rows (see gru_recur_unit_kernel): sequence b's gi rows start at GI + row0[b] * ldg,
// only h at t = T-1 is stored, to out [B][H]
template <bool SAVE, int NB, int KPT, bool WIN = false>
__global__ void __launch_bounds__(kRwThreads, 1)
    gru_recur_regw_kernel(const float* __restrict__ GI, const float* __restrict__ WhT, const float* __restrict__ bhn,
                          float* __restrict__ out, long long B, int T, int H, int ldg, int NP, float* __restrict__ gsave,
                          int ldsave, const long long* __restrict__ row0) {
    extern __shared__ __align__(16) float smem[];
    constexpr int RS = KPT + 4;
    float* hs = smem;                          // [4][RS]
    float* gis = hs + kRsBT * RS;              // [2][4][ldg]
    float* ghs = gis + 2 * kRsBT * ldg;        // [4][NP]
    float* bns = ghs + kRsBT * NP;             // [KPT]
    const int tid = threadIdx.x;
    const long long b0 = (long long)blockIdx.x * kRsBT;
    const int H2 = 2 * H;

    // this thread's gate column of W_hh^T ([KPT][NP], zero padded): registers for the whole kernel
    const bool gemm_thread = tid < NP;
    float w[KPT];
#pragma unroll
    for (int k = 0; k < KPT; ++k) w[k] = gemm_thread ? __ldg(WhT + (size_t)k * NP + tid) : 0.0f;

    for (int e = tid; e < kRsBT * RS; e += kRwThreads) hs[e] = 0.0f;
    for (int e = tid; e < 2 * kRsBT * ldg; e += kRwThreads) gis[e] = 0.0f;
    for (int e = tid; e < kRsBT * NP; e += kRwThreads) ghs[e] = 0.0f;
    for (int e = tid; e < KPT; e += kRwThreads) bns[e] = e < H ? __ldg(bhn + e) : 0.0f;

    // gi rows of step t -> buffer (t & 1): each thread owns fixed 16-byte chunks whose source advances one row per step
    const int chunks = ldg >> 2;
    constexpr int kPfMax = (kRsBT * (4 * 128) / 4 + kRwThreads - 1) / kRwThreads;
    const float* pf_src[kPfMax];
    int pf_off[kPfMax];       // float offset inside a gi buffer, -1: no chunk
    bool pf_ok[kPfMax];
#pragma unroll
    for (int q = 0; q < kPfMax; ++q) {
        const int e = tid + q * kRwThreads;
        const bool mine = e < kRsBT * chunks;
        const int b = mine ? e / chunks : 0, c = mine ? e - b * chunks : 0;
        pf_ok[q] = mine && (b0 + b < B);
        pf_off[q] = mine ? b * ldg + 4 * c : -1;
        pf_src[q] = WIN ? GI + (size_t)(pf_ok[q] ? row0[b0 + b] : 0) * ldg + 4 * c
                        : GI + ((size_t)(pf_ok[q] ? b0 + b : 0) * T) * ldg + 4 * c;
    }
#define WG_RW_PREFETCH(t_)                                                                              \
    do {                                                                                                \
        float* dstb_ = gis + ((t_) & 1) * kRsBT * ldg;                                                  \
        _Pragma("unroll") for (int q = 0; q < kPfMax; ++q)                                              \
            if (pf_off[q] >= 0) cp_async16(dstb_ + pf_off[q], pf_src[q] + (size_t)(t_) * ldg, pf_ok[q]); \
        cp_async_commit();                                                                              \
    } while (0)
    __syncthreads();
    WG_RW_PREFETCH(0);

    const int nb = (int)((B - b0) < kRsBT ? (B - b0) : kRsBT);   // sequences of this CTA that exist

    for (int t = 0; t < T; ++t) {
        if (t + 1 < T) WG_RW_PREFETCH(t + 1);
        const float* g = gis + (t & 1) * kRsBT * ldg;
        if (t > 0 && gemm_thread) {   // h_{-1} = 0: the product is zero at t == 0 (ghs was zeroed above)
            float acc[NB];
#pragma unroll
            for (int i = 0; i < NB; ++i) acc[i] = 0.0f;
#pragma unroll
            for (int k = 0; k < KPT; k += 4) {
#pragma unroll
                for (int i = 0; i < NB; ++i) {
                    const float4 h = *reinterpret_cast<const float4*>(hs + i * RS + k);
                    acc[i] = fmaf(h.x, w[k], acc[i]);
                    acc[i] = fmaf(h.y, w[k + 1], acc[i]);
                    acc[i] = fmaf(h.z, w[k + 2], acc[i]);
                    acc[i] = fmaf(h.w, w[k + 3], acc[i]);
                }
            }
#pragma unroll
            for (int i = 0; i < NB; ++i) ghs[i * NP + tid] = acc[i];
        }
        if (t + 1 < T) cp_async_wait<1>(); else cp_async_wait<0>();
        __syncthreads();   // gi(t) and gh(t) complete
#pragma unroll
        for (int u = 0; u < (kRsBT * 128 + kRwThreads - 1) / kRwThreads; ++u) {
            const int e = tid + u * kRwThreads;
            if (e < nb * H) {
                const int b = e / H, j = e - b * H;
                const float* gr = g + b * ldg + j;
                const float* gh = ghs + b * NP + j;
                const float r = sigmoid_f(gr[0] + gh[0]);
                const float z = sigmoid_f(gr[H] + gh[H]);
                const float hn = gh[H2] + bns[j];
                const float n = tanh_f(gr[H2] + r * hn);
                const float hnew = (hs[b * RS + j] - n) * z + n;
                hs[b * RS + j] = hnew;
                if (WIN) {
                    if (b0 + b < B && t == T - 1) out[(size_t)(b0 + b) * H + j] = hnew;
                } else if (b0 + b < B) {
                    out[((size_t)(b0 + b) * T + t) * H + j] = hnew;
                    if (SAVE) {
                        float* gs = gsave + ((size_t)(b0 + b) * T + t) * ldsave + j;
                        gs[0] = r;
                        gs[H] = z;
                        gs[H2] = n;
                        gs[H2 + H] = hn;
                    }
                }
            }
        }
        __syncthreads();   // h(t) visible before the next product; gi buffer (t & 1) and gh free again
    }
#undef WG_RW_PREFETCH
}

}  // namespace wg
