// GRU recurrence on the 5th-generation tensor cores (tcgen05): the tensor-path counterpart of
// recur_unit.cuh, selected by WG_FLAG_TENSOR_CORES.
//
// Reference: `gru_out, _ = self.gru(hidden2)` at src/step6_gcn_gru_combined_model.py:23 (module
// built at :11); gate equations in recur.cuh.
//
// Per step the recurrent product  gh[n][c] = sum_k W_hh[c][k] * h[n][k]  is issued as
//     D[c][n] = A[c][k] . B[n][k]^T,   A = W_hh (one 128-row tile per gate, rows = hidden units),
//                                       B = h of the group's N = 16 sequences,  K = H padded to 16
// with both operands split into two fp16 parts, x = hi + lo (hi = fp16(x), lo = fp16(x - hi): 22
// significant bits, and fp16 x fp16 products are exact in the fp32 accumulator):
//     D ~= A_hi.B_hi + A_hi.B_lo + A_lo.B_hi          (kind::f16, M = 128, N = 16, K = 16)
// Both operands are scaled by powers of two before the split (tc_scale_exp: a W_hh row by its own exponent, h by
// the fixed 2^kTcHExp) and the gate phase undoes both with one factor per gate and hidden unit, so the split keeps
// its 22 bits whatever the magnitude of W_hh or h.
// The A_hi.B_hi products go to one TMEM accumulator, the two corrections to a second one (TMEM
// accumulation truncates — tcgen05.cuh — so the small terms are kept apart from the big ones and the
// two are added with round-to-nearest in the epilogue).  The dropped lo.lo term is 2^-22 relative.
//
// Why this layout: with the hidden unit on the M axis, TMEM lane j of all three gate tiles holds
// gh_r[j], gh_z[j], gh_n[j] of a sequence in ONE thread — the gate math needs no exchange at all —
// and a warp's stores of h_t (global, [b][t][j]) and loads of gi ([b*T + t][g*H + j]) are contiguous
// along j.  The new state goes back to shared memory as the next step's B operand (fp16 hi / lo,
// UMMA canonical K-major layout, 2-byte stores; the 16-byte K chunks are 16 bytes further apart than
// they need to be so that the four chunks a warp writes hit different banks).
//
// A CTA holds W_hh (hi + lo, 172 KB at H = 102) in shared memory and runs two independent groups of 16
// sequences.  A group = 8 warps: warps 0-3 (TMEM lanes 0..127 = hidden units) take its sequences 0-7,
// warps 4-7 its sequences 8-15.  Per step the group's warps do the gate math, write h_t, meet at a named
// barrier, three threads of the group (one per gate tile) issue the 42 MMAs of the next step and commit them
// to the group's mbarrier, on which all eight warps then wait (their next gi values are already in flight).  The two
// groups never synchronise with each other, so one group's product (tensor pipe) overlaps the other's
// gate math (MUFU / ALU).  The hi.hi and hi.lo products share one N = 32 MMA (B rows = h_hi | h_lo), so
// A_hi is read from shared memory once for both.
//
// The same kernel serves every batch size in the tensor path (a result never depends on how a batch
// is split: the columns of an MMA are independent).
#pragma once

#include <cuda_fp16.h>

#include "recur.cuh"
#include "tcgen05.cuh"
#include "wg_common.cuh"

namespace wg {

constexpr int kRtN = 16;        // sequences per group
constexpr int kRtGroups = 2;    // groups per CTA
constexpr int kRtGroupWarps = 8;          // warps per group: two sets of 4 (TMEM lane quarters), 8 sequences each
constexpr int kRtThreads = kRtGroups * kRtGroupWarps * 32;
constexpr int kRtSeqs = kRtN * kRtGroups;
// B operand of a group: rows 0..15 = h_hi of its sequences, rows 16..31 = h_lo; 16-byte K chunks are
// (32 rows + 1) * 16 bytes apart (the extra 16 bytes spread the chunks a warp writes over the banks)
constexpr int kRtBLbo = 2 * kRtN * 16 + 16;

__host__ __device__ inline int recur_tc_kp(int H) { return round_up(H, 16); }
__host__ __device__ inline bool recur_tc_applies(int H) { return H <= 128; }
// halves of one part (hi or lo) of the packed W_hh: [3 gates][KP/8 chunks][128 rows][8]
__host__ __device__ inline size_t recur_tc_w_halves(int H) { return (size_t)3 * (recur_tc_kp(H) / 8) * 128 * 8; }
__host__ __device__ inline size_t recur_tc_smem_bytes(int H) {
    const int nch = recur_tc_kp(H) / 8;
    size_t n = 2 * recur_tc_w_halves(H) * 2;                    // A hi + lo
    n += (size_t)kRtGroups * nch * kRtBLbo;                     // B (hi and lo rows) per group
    n += 64;                                                    // mbarriers, TMEM slot
    return n + 128;                                             // alignment slack
}

__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
    // D = F32 (1 at bit 4), A = B = F16 (0 at bits 7 and 10), both K-major, N >> 3 at [17,23), M >> 4 at [24,29)
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// wait for the outstanding tcgen05.ld's; the loaded registers are operands so that no use can move above the wait
__device__ __forceinline__ void tmem_ld_wait(float (&v)[8]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;\n"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7])
                 :
                 : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// Power-of-two scales of the split fp16 operands.  Unscaled, lo = fp16(x - hi) is an fp16 subnormal below |x| = 2^-3
// (a fixed absolute error of 2^-25, so the relative precision falls with the magnitude) and hi overflows above 65504.
// A row whose largest magnitude is m is multiplied by 2^e with m 2^e in [2^14, 2^15) before the split and the
// product by 2^-e after it, in fp32: every element down to 2^-17 m keeps 22 significant bits, at any m, and a row
// rescaled by a power of two splits into exactly rescaled parts.  e is clamped to [-kTcExpMax, kTcExpMax] so that
// the product of two inverse factors is a normal fp32; a zero, infinite or NaN m gets e = 0.
constexpr int kTcExpMax = 63;
constexpr int kTcHExp = 14;   // the GRU state: |h| < 1, a fixed 2^14
__device__ __forceinline__ int tc_scale_exp(float m) {
    if (!(m > 0.0f) || !(m <= 3.402823466e38f)) return 0;
    int E;
    frexpf(m, &E);   // m = f 2^E, f in [0.5, 1)
    const int e = 15 - E;
    return e < -kTcExpMax ? -kTcExpMax : (e > kTcExpMax ? kTcExpMax : e);
}
__device__ __forceinline__ float tc_exp2(int e) { return __int_as_float((127 + e) << 23); }   // e in [-126, 127]
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// w_hh [3H][H] fp32 -> hi / lo fp16 parts in the UMMA K-major layout [gate][k / 8][128 rows][k % 8], each row
// (gate g, hidden unit j) scaled by 2^e(row) before the split; funit [3][128] = 2^-(e(row) + kTcHExp), the factor
// that undoes the row's and h's scales.  One warp per row.
__global__ void pack_whh_tc_kernel(const float* __restrict__ w_hh, __half* __restrict__ hi, __half* __restrict__ lo,
                                   float* __restrict__ funit, int H) {
    const int nch = recur_tc_kp(H) / 8, KP = nch * 8, lane = threadIdx.x & 31;
    const int nwarps = gridDim.x * blockDim.x / 32;
    for (int row = (blockIdx.x * blockDim.x + threadIdx.x) / 32; row < 3 * 128; row += nwarps) {
        const int g = row / 128, j = row % 128;
        const float* w = w_hh + ((size_t)g * H + (j < H ? j : 0)) * H;
        float m = 0.0f;
        if (j < H)
            for (int k = lane; k < H; k += 32) m = fmaxf(m, fabsf(w[k]));
        const int e = tc_scale_exp(warp_max(m));
        const float sc = tc_exp2(e);
        if (lane == 0) funit[row] = tc_exp2(-e - kTcHExp);
        for (int k = lane; k < KP; k += 32) {
            const float v = (j < H && k < H) ? w[k] * sc : 0.0f;
            const size_t idx = (((size_t)g * nch + k / 8) * 128 + j) * 8 + k % 8;
            const __half h = __float2half_rn(v);
            hi[idx] = h;
            lo[idx] = __float2half_rn(v - __half2float(h));
        }
    }
}

// GI [rows][ldg] (b_ih, and b_hh of r / z, folded in; readable up to the next multiple of kRtSeqs sequences);
// Whi / Wlo / funit: pack_whh_tc_kernel's output; out [B][T][H]
// WIN: windows over one table's gi rows (see gru_recur_unit_kernel): sequence b's gi rows start at GI + row0[b] * ldg
// (the padding sequences of the last group read the last window's rows), only h at t = T-1 is stored, to out [B][H]
template <bool WIN = false>
__global__ void __launch_bounds__(kRtThreads, 1)
    gru_recur_tc_kernel(const float* __restrict__ GI, const __half* __restrict__ Whi, const __half* __restrict__ Wlo,
                        const float* __restrict__ funit, const float* __restrict__ bhn, float* __restrict__ out,
                        long long B, int T, int H, int ldg, const long long* __restrict__ row0) {
    extern __shared__ __align__(1024) unsigned char smem_rt[];
    const int KP = recur_tc_kp(H), NCH = KP / 8, NKS = KP / 16;
    const uint32_t a_part = (uint32_t)(3 * NCH * 2048);           // bytes of A_hi (= A_lo)
    const uint32_t b_grp = (uint32_t)(NCH * kRtBLbo);             // bytes of one group's B operand
    unsigned char* sA = smem_rt;                                   // [hi | lo][gate][chunk][128][8 halves]
    unsigned char* sB = sA + 2 * a_part;                           // [group][chunk][hi rows | lo rows][8 halves]
    uint64_t* acc_full = reinterpret_cast<uint64_t*>(sB + kRtGroups * b_grp);        // [groups]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + kRtGroups);

    const int tid = threadIdx.x, warp = tid >> 5;
    const long long b0 = (long long)blockIdx.x * kRtSeqs;

    // ---- stage W_hh (hi, lo) and zero the state operand ----
    {
        const uint4* s0 = reinterpret_cast<const uint4*>(Whi);
        const uint4* s1 = reinterpret_cast<const uint4*>(Wlo);
        uint4* d = reinterpret_cast<uint4*>(sA);
        const int n16 = (int)(a_part / 16);
        for (int e = tid; e < n16; e += kRtThreads) {
            d[e] = __ldg(s0 + e);
            d[n16 + e] = __ldg(s1 + e);
        }
        uint32_t* z = reinterpret_cast<uint32_t*>(sB);
        for (int e = tid; e < (int)(kRtGroups * b_grp / 4); e += kRtThreads) z[e] = 0u;
    }
    if (tid == 0) {
        for (int g = 0; g < kRtGroups; ++g) mbar_init(&acc_full[g], 3);   // one commit per gate tile
        fence_mbar_init();
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)),
                     "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    fence_async_smem();   // the staged operands (generic-proxy writes) are read by the tensor core (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // TMEM columns of group g start at g * 6N; gate q: [q * 2N, q * 2N + N) = hi.hi, [q * 2N + N, q * 2N + 2N) =
    // the corrections.  One N = 32 MMA (B rows = h_hi | h_lo) writes both with a single read of A_hi; the
    // lo.hi product (A_lo, B rows = h_hi, N = 16) is accumulated onto the correction columns.

    const int g = warp / kRtGroupWarps;                   // group of this warp
    const int gt = tid - g * kRtGroupWarps * 32;          // thread index inside the group, 0 .. 255
    const int half = gt >> 7;                             // sequences 8 half .. 8 half + 7 of the group
    const int j = gt & 127;                               // hidden unit = TMEM lane
    const bool unit_ok = j < H;
    const int jc = unit_ok ? j : H - 1;
    const float bn = __ldg(bhn + jc);
    const float fr = __ldg(funit + jc), fz = __ldg(funit + 128 + jc), fn = __ldg(funit + 256 + jc);   // 2^-(e + 14)
    const uint32_t tcol = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(g * 6 * kRtN + half * 8);
    // byte address of this unit inside the group's B operand: chunk j / 8, element j % 8 (row n adds n * 16)
    unsigned char* bh = sB + (size_t)g * b_grp + (size_t)(jc >> 3) * kRtBLbo + (size_t)(jc & 7) * 2 + half * 8 * 16;
    unsigned char* bl = bh + kRtN * 16;
    float hprev[8];
#pragma unroll
    for (int n = 0; n < 8; ++n) hprev[n] = 0.0f;
    const int H2 = 2 * H;
    const long long bg0 = b0 + g * kRtN + half * 8;       // first sequence of this thread
    const long long left = B - bg0;
    const int nvalid = left >= 8 ? 8 : (left > 0 ? (int)left : 0);
    // running pointers (advance one step at a time); sequences are T * ldg / T * H floats apart
    // (WIN: out rows H floats apart, written at the last step; gi rows from gw)
    const float* gp = GI + (size_t)bg0 * T * ldg + jc;
    float* op = out + (size_t)bg0 * (WIN ? 1 : T) * H + j;
    const int g_seq = T * ldg, o_seq = (WIN ? 1 : T) * H;
    const float* gw[WIN ? 8 : 1];
    if (WIN) {
#pragma unroll
        for (int n = 0; n < (WIN ? 8 : 1); ++n) gw[n] = GI + (size_t)row0[bg0 + n < B ? bg0 + n : B - 1] * ldg + jc;
    }
    uint32_t ph = 0;
    // MMA issue (one thread per group): operand bases
    const uint32_t idesc32 = umma_idesc_f16(128, 2 * kRtN), idesc16 = umma_idesc_f16(128, kRtN);
    const uint32_t sa = smem_u32(sA), sbg = smem_u32(sB) + (uint32_t)g * b_grp;
    const uint32_t dcol = tmem_base + (uint32_t)(g * 6 * kRtN);

    // gi of this thread's 8 sequences: [gate][seq]; rows beyond B are readable scratch (never stored)
    // (WIN: step t of sequence n at gw[n] + t * ldg)
    auto load_gi = [&](float (&gi)[3][8], const float* p, int t) {
#pragma unroll
        for (int n = 0; n < 8; ++n) {
            const float* s = WIN ? gw[WIN ? n : 0] + (size_t)t * ldg : p + n * g_seq;
            gi[0][n] = __ldg(s);
            gi[1][n] = __ldg(s + H);
            gi[2][n] = __ldg(s + H2);
        }
    };
    float gi[3][8], gi_nxt[3][8];
    load_gi(gi, gp, 0);
    for (int t = 0; t < T; ++t) {
        if (t + 1 < T) load_gi(gi_nxt, gp + ldg, t + 1);   // a whole step ahead: lands during this step's gates + product
        float rr[8], zz[8], hn[8];
        if (t > 0) {
            mbar_wait(&acc_full[g], ph);   // this group's product of step t is complete
            ph ^= 1;
            tc_fence_after();
            float m[8], c[8];
            tmem_ld8(tcol, m);
            tmem_ld8(tcol + kRtN, c);
            tmem_ld_wait(m);
            tmem_ld_wait(c);
#pragma unroll
            for (int n = 0; n < 8; ++n) rr[n] = fmaf(m[n] + c[n], fr, gi[0][n]);
            tmem_ld8(tcol + 2 * kRtN, m);
            tmem_ld8(tcol + 3 * kRtN, c);
            tmem_ld_wait(m);
            tmem_ld_wait(c);
#pragma unroll
            for (int n = 0; n < 8; ++n) zz[n] = fmaf(m[n] + c[n], fz, gi[1][n]);
            tmem_ld8(tcol + 4 * kRtN, m);
            tmem_ld8(tcol + 5 * kRtN, c);
            tmem_ld_wait(m);
            tmem_ld_wait(c);
#pragma unroll
            for (int n = 0; n < 8; ++n) hn[n] = fmaf(m[n] + c[n], fn, bn);
            tc_fence_before();   // the accumulators have been read: the next product may overwrite them
        } else {
#pragma unroll
            for (int n = 0; n < 8; ++n) {
                rr[n] = gi[0][n];
                zz[n] = gi[1][n];
                hn[n] = bn;
            }
        }
#pragma unroll
        for (int n = 0; n < 8; ++n) {
            const float r = sigmoid_f(rr[n]);
            const float z = sigmoid_f(zz[n]);
            const float nv = tanh_f(gi[2][n] + r * hn[n]);
            const float hnew = (hprev[n] - nv) * z + nv;
            hprev[n] = hnew;
            if (unit_ok) {
                const float hs = hnew * (float)(1 << kTcHExp);
                const __half hh = __float2half_rn(hs);
                const __half hl = __float2half_rn(hs - __half2float(hh));
                *reinterpret_cast<__half*>(bh + n * 16) = hh;
                *reinterpret_cast<__half*>(bl + n * 16) = hl;
                if (n < nvalid && (!WIN || t == T - 1)) op[n * o_seq] = hnew;
            }
        }
        gp += ldg;
        if (!WIN) op += H;
        if (t + 1 < T) {
            // h_t of the group is in shared memory (generic-proxy writes -> visible to the tensor core), every
            // warp of the group has read its accumulators: one thread issues the next step's product
            fence_async_smem();
            group_barrier(1 + g, kRtGroupWarps * 32);
            if ((gt & 31) == 0 && gt < 96) {
                // three issuing threads per group (lane 0 of its warps 0, 1, 2), one gate tile each: the 14 MMAs of
                // a gate are issued back to back (descriptors advance by constant increments) and committed to
                // the group's mbarrier, which completes when all three commits have
                tc_fence_after();
                const int q = gt >> 5;
                uint64_t da_hi = umma_desc_kmajor(sa + (uint32_t)q * NCH * 2048, 2048, 128);
                uint64_t da_lo = umma_desc_kmajor(sa + a_part + (uint32_t)q * NCH * 2048, 2048, 128);
                uint64_t db = umma_desc_kmajor(sbg, kRtBLbo, 128);
                const uint32_t d0 = dcol + q * 2 * kRtN;
                for (int ks = 0; ks < NKS; ++ks) {
                    umma_f16(d0, da_hi, db, idesc32, ks != 0);            // hi.hi | hi.lo
                    umma_f16(d0 + kRtN, da_lo, db, idesc16, 1);           // lo.hi
                    da_hi += (2 * 2048) >> 4;                             // start-address field: 16-byte units
                    da_lo += (2 * 2048) >> 4;
                    db += (2 * kRtBLbo) >> 4;
                }
                umma_commit(&acc_full[g]);
            }
#pragma unroll
            for (int q = 0; q < 3; ++q)
#pragma unroll
                for (int n = 0; n < 8; ++n) gi[q][n] = gi_nxt[q][n];
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512));
    }
}

}  // namespace wg
