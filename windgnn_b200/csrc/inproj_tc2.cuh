// GRU input projection on tcgen05, second generation: fp16 split operands, U read ONCE as fp32.
//     GI = U . W_ih^T + b,   x = hi + lo with hi = fp16(x), lo = fp16(x - hi)   (22 significant bits)
//     U.W ~= U_hi.W_hi + U_hi.W_lo + U_lo.W_hi        (kind::f16: fp16 x fp16 products are exact in the
//                                                      fp32 accumulator; the dropped lo.lo term is 2^-22)
// Before the split each U row and each W_ih row (gate column) is scaled by a power of two (tc_scale_exp, recur_tc.cuh)
// that maps its largest magnitude into [2^14, 2^15); the epilogue undoes both with one factor per output,
//     GI[r][c] = (acc_hi + acc_corr) * 2^-(e_r + e_c) + b[c],
// so the relative error of the split does not depend on the scale of U or W_ih and no operand leaves the fp16 range.
// The largest element of each U row (U >= 0 after the ReLU: float bits compare as integers) is recorded in umax by
// the GCN kernel that writes the row, or by u_rowmax_kernel.
//
// Reference: the `gi = W_ih u + b_ih` half of nn.GRU, src/step6_gcn_gru_combined_model.py:11,23.
//
// The first-generation kernel (kind::tf32, hi / lo copies of both operands in HBM) moved 11.1 GB from L2
// for 2.06 GB of algorithmic operand bytes and was L2-bound with the tensor pipe 49 % busy (ncu r01).
// Here the GCN kernel's ordinary fp32 tiles are the A operand: a stage's [32 k][128 rows] fp32 block
// arrives by one bulk copy, four converter warps split it into fp16 hi / lo in the UMMA K-major layout
// in shared memory (never in HBM), and kind::f16 halves both the operand bytes and the MMA time of
// kind::tf32.  W_ih is pre-split once per call (pack kernel) and streamed from L2 one stage at a time.
//
// One persistent CTA per SM, 14 warps:
//   warp 12      producer: per stage two bulk async copies (A fp32 16 KB, B hi+lo 20 KB at N = 160)
//   warps 8-11   converters: a thread takes 2 rows x 8 k's (8-byte loads), scales them by 2^e_r, splits fp32 -> fp16 hi / lo and
//                writes 16-byte chunks into the canonical layout ([k / 8][row][8 halves]: 8-row x 16-byte
//                core matrices, SBO = 128 B, LBO = rows * 16 B)
//   warp 13      MMA issuer: 6 x tcgen05.mma.kind::f16 (M = 128, N <= 160, K = 16) per stage;
//                hi.hi into one TMEM accumulator, the corrections into a second one (TMEM accumulation
//                truncates: the small terms are kept apart and added in fp32 in the epilogue)
//   warps 0-7    epilogue: warp w reads TMEM lanes 32 (w % 4) .. and the column half w / 4: tcgen05.ld, sum,
//                x 2^-(e_r + e_c) + bias (one FMA), 32-byte stores (GI rows are 32-byte aligned); the accumulators are released to the
//                issuer as soon as a warp's last block is in registers
#pragma once

#include <cuda_fp16.h>

#include "recur_tc.cuh"
#include "tcgen05.cuh"
#include "wg_common.cuh"

namespace wg {

constexpr int kT2BM = 128;
constexpr int kT2BK = 32;                 // k's per pipeline stage (two MMA k-steps)
constexpr int kT2EpiWarps = 8;            // two per TMEM lane quarter: each takes half of the tile's columns
constexpr int kT2ConvWarps = 4;
constexpr int kT2Threads = (kT2EpiWarps + kT2ConvWarps + 2) * 32;   // epilogue, converters, producer, MMA issuer
constexpr int kT2MaxN = 160;              // gate columns per CTA tile (two accumulators of N columns in TMEM)

struct Tc2Shape {
    int NP;        // padded gate columns = n_nt * N_each
    int n_nt;      // column slices
    int N_each;    // MMA N (multiple of 16)
    int KP;        // K rounded up to kT2BK
    int stages;
    size_t stage_bytes, smem_bytes;
    bool ok;
};

__host__ inline Tc2Shape tc2_shape(int G, int I) {
    Tc2Shape s{};
    const int np16 = round_up(G, 16);
    s.n_nt = ceil_div(np16, kT2MaxN);
    s.N_each = round_up(ceil_div(np16, s.n_nt), 16);
    s.NP = s.n_nt * s.N_each;
    s.KP = round_up(I, kT2BK);
    // A fp32 block + A hi/lo fp16 + B hi/lo fp16
    s.stage_bytes = (size_t)kT2BM * kT2BK * 4 + (size_t)2 * kT2BM * kT2BK * 2 + (size_t)2 * s.N_each * kT2BK * 2;
    s.stages = (int)((kMaxSmemOptin - 1024) / s.stage_bytes);
    if (s.stages > 6) s.stages = 6;
    s.ok = s.N_each <= kT2MaxN && s.stages >= 2;
    s.smem_bytes = s.stage_bytes * s.stages + 1024;
    return s;
}
// halves of the packed W_ih (hi and lo together): [n_nt][KP / 32 stages][hi | lo][4 chunks][N_each][8]
__host__ inline size_t tc2_w_halves(const Tc2Shape& s) { return (size_t)2 * s.NP * s.KP; }

// w_ih [G][I] fp32 -> per (column slice, stage) one contiguous block [hi | lo][k chunk][n][8 halves], gate column n
// scaled by 2^e(n) before the split; colinv [NP] = 2^-e(n).  One warp per gate column.
__global__ void pack_wih_tc2_kernel(const float* __restrict__ w_ih, __half* __restrict__ wp, float* __restrict__ colinv,
                                    int G, int I, int KP, int n_nt, int N_each) {
    const int nst = KP / kT2BK, NP = n_nt * N_each, lane = threadIdx.x & 31;
    const int nwarps = gridDim.x * blockDim.x / 32;
    for (int n = (blockIdx.x * blockDim.x + threadIdx.x) / 32; n < NP; n += nwarps) {
        const float* w = w_ih + (size_t)(n < G ? n : 0) * I;
        float m = 0.0f;
        if (n < G)
            for (int k = lane; k < I; k += 32) m = fmaxf(m, fabsf(w[k]));
        const int e = tc_scale_exp(warp_max(m));
        const float sc = tc_exp2(e);
        if (lane == 0) colinv[n] = tc_exp2(-e);
        const int nt = n / N_each, nl = n % N_each;
        for (int k = lane; k < KP; k += 32) {
            const float v = (n < G && k < I) ? w[k] * sc : 0.0f;
            // [nt][k / 32][part][k % 32 / 8][nl][k % 8]; the lo part is 4 chunks further
            const size_t idx = ((((size_t)nt * nst + k / kT2BK) * 2 * 4 + (k % kT2BK) / 8) * N_each + nl) * 8 + k % 8;
            const __half h = __float2half_rn(v);
            wp[idx] = h;
            wp[idx + (size_t)4 * N_each * 8] = __float2half_rn(v - __half2float(h));
        }
    }
}

// umax[r] = the largest element of U row r (>= 0: float bits), for whole 128-row tiles (0 past `rows`); for the GCN
// kernels that do not record it while they write U.  A thread per row: a warp reads 128 contiguous bytes per k.
__global__ void __launch_bounds__(256) u_rowmax_kernel(const float* __restrict__ U, int* __restrict__ umax,
                                                       long long rows, int ldk) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= (rows + kT2BM - 1) / kT2BM * kT2BM) return;
    float m = 0.0f;
    if (r < rows) {
        const float* u = U + (size_t)(r / kT2BM) * ldk * kT2BM + r % kT2BM;
#pragma unroll 8
        for (int k = 0; k < ldk; ++k) m = fmaxf(m, __ldg(u + (size_t)k * kT2BM));
    }
    umax[r] = __float_as_int(m);
}

// A: U tiles [M/128][lda][128] fp32 (lda >= KP, K-major 128-row tiles written by the GCN kernels);
// umax: [whole tiles of M rows] row maxima (float bits); Wp, colinv: pack_wih_tc2_kernel's output;
// C: [M][ldc] row-major (GI)
__global__ void __launch_bounds__(kT2Threads, 1)
    inproj_tc2_kernel(const float* __restrict__ A, const int* __restrict__ umax, const __half* __restrict__ Wp,
                      const float* __restrict__ colinv, const float* __restrict__ bias, float* __restrict__ C,
                      long long M, int lda, int KP, int ldc, int n_nt, int N_each, int stages) {
    extern __shared__ __align__(1024) unsigned char smem_t2[];
    const uint32_t a32_bytes = kT2BM * kT2BK * 4;                   // 16 KB
    const uint32_t a16_bytes = kT2BM * kT2BK * 2;                   // 8 KB per part
    const uint32_t b_bytes = (uint32_t)N_each * kT2BK * 2;          // per part
    const uint32_t stage_bytes = a32_bytes + 2 * a16_bytes + 2 * b_bytes;
    unsigned char* tail = smem_t2 + (size_t)stage_bytes * stages;
    uint64_t* full_ld = reinterpret_cast<uint64_t*>(tail);           // [stages] bulk copies landed
    uint64_t* full_cv = full_ld + 8;                                  // [stages] A converted
    uint64_t* empty_bar = full_cv + 8;                                // [stages] MMAs have read the stage
    uint64_t* tmem_full = empty_bar + 8;
    uint64_t* tmem_empty = tmem_full + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long m_tiles = (M + kT2BM - 1) / kT2BM;
    const long long n_tiles = m_tiles * n_nt;   // tile = mt * n_nt + nt: the slices of one row tile run together
    const int KB = KP / kT2BK;

    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_ld[s], 1);
            mbar_init(&full_cv[s], kT2ConvWarps);   // one arrival per converter warp
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, kT2EpiWarps);   // one arrival per epilogue warp
        fence_mbar_init();
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)),
                     "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t acc_cols = (uint32_t)N_each;   // accumulators: [0, N) hi.hi, [N, 2N) corrections

    if (warp == kT2EpiWarps + kT2ConvWarps) {
        // ===================== producer =====================
        int s = 0;
        uint32_t phase = 0;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const long long mt = tile / n_nt;
            const int nt = (int)(tile - mt * n_nt);
            const float* a = A + (size_t)mt * lda * kT2BM;
            const __half* b = Wp + (size_t)nt * KB * 2 * N_each * kT2BK;
            for (int kb = 0; kb < KB; ++kb) {
                if (lane == 0) {
                    mbar_wait(&empty_bar[s], phase ^ 1);  // slot free (first pass: passes immediately)
                    unsigned char* st = smem_t2 + (size_t)s * stage_bytes;
                    mbar_expect_tx(&full_ld[s], a32_bytes + 2 * b_bytes);
                    bulk_g2s(st, a + (size_t)kb * kT2BK * kT2BM, a32_bytes, &full_ld[s]);
                    bulk_g2s(st + a32_bytes + 2 * a16_bytes, b + (size_t)kb * 2 * N_each * kT2BK, 2 * b_bytes,
                             &full_ld[s]);
                }
                __syncwarp();
                if (++s == stages) { s = 0; phase ^= 1; }
            }
        }
    } else if (warp >= kT2EpiWarps && warp < kT2EpiWarps + kT2ConvWarps) {
        // ===================== converters: item = (row pair, 8-k chunk), two items per thread and stage ==========
        const int ct = tid - kT2EpiWarps * 32;    // 0 .. 127
        int s = 0;
        uint32_t phase = 0;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            // this thread's rows 2 rp, 2 rp + 1 (rp = ct % 64 for both items): their scales 2^e_r
            const long long r0 = tile / n_nt * kT2BM + 2 * (ct & 63);
            const float sc0 = tc_exp2(tc_scale_exp(__int_as_float(__ldg(umax + r0))));
            const float sc1 = tc_exp2(tc_scale_exp(__int_as_float(__ldg(umax + r0 + 1))));
            for (int kb = 0; kb < KB; ++kb) {
                mbar_wait(&full_ld[s], phase);
                unsigned char* st = smem_t2 + (size_t)s * stage_bytes;
#pragma unroll
                for (int it = 0; it < (kT2BM / 2) * (kT2BK / 8) / (kT2ConvWarps * 32); ++it) {
                    const int item = ct + it * kT2ConvWarps * 32;
                    const int rp = item & 63, c = item >> 6;      // rows 2 rp, 2 rp + 1; k's 8 c .. 8 c + 7 of the stage
                    const float* a32 = reinterpret_cast<const float*>(st) + (c * 8) * kT2BM + 2 * rp;   // [k][128 rows]
                    unsigned char* hi = st + a32_bytes + c * (kT2BM * 16) + (2 * rp) * 16;             // [chunk][row][8 halves]
                    unsigned char* lo = hi + a16_bytes;
                    float2 v[8];
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk) {
                        v[kk] = *reinterpret_cast<const float2*>(a32 + kk * kT2BM);
                        v[kk].x *= sc0;
                        v[kk].y *= sc1;
                    }
                    __half2 h0[4], l0[4], h1[4], l1[4];   // row 2 rp / row 2 rp + 1: k pairs
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        h0[q] = __floats2half2_rn(v[2 * q].x, v[2 * q + 1].x);
                        h1[q] = __floats2half2_rn(v[2 * q].y, v[2 * q + 1].y);
                        const float2 b0 = __half22float2(h0[q]), b1 = __half22float2(h1[q]);
                        l0[q] = __floats2half2_rn(v[2 * q].x - b0.x, v[2 * q + 1].x - b0.y);
                        l1[q] = __floats2half2_rn(v[2 * q].y - b1.x, v[2 * q + 1].y - b1.y);
                    }
                    *reinterpret_cast<uint4*>(hi) = *reinterpret_cast<uint4*>(h0);
                    *reinterpret_cast<uint4*>(hi + 16) = *reinterpret_cast<uint4*>(h1);
                    *reinterpret_cast<uint4*>(lo) = *reinterpret_cast<uint4*>(l0);
                    *reinterpret_cast<uint4*>(lo + 16) = *reinterpret_cast<uint4*>(l1);
                }
                fence_async_smem();   // the converted operand is read by the tensor core (async proxy)
                __syncwarp();
                if (lane == 0) mbar_arrive(&full_cv[s]);
                if (++s == stages) { s = 0; phase ^= 1; }
            }
        }
    } else if (warp == kT2EpiWarps + kT2ConvWarps + 1) {
        // ===================== MMA issuer =====================
        const uint32_t idesc = umma_idesc_f16(kT2BM, N_each);
        const uint32_t lbo_a = kT2BM * 16, lbo_b = (uint32_t)N_each * 16, sbo = 128;
        int s = 0;
        uint32_t phase = 0, acc_phase = 0;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            if (lane == 0) {
                mbar_wait(tmem_empty, acc_phase ^ 1);  // epilogue has drained the accumulators
                tc_fence_after();
            }
            __syncwarp();
            for (int kb = 0; kb < KB; ++kb) {
                if (lane == 0) {
                    mbar_wait(&full_ld[s], phase);     // B landed (async proxy)
                    mbar_wait(&full_cv[s], phase);     // A converted
                    tc_fence_after();
                    const uint32_t st = smem_u32(smem_t2 + (size_t)s * stage_bytes);
                    const uint32_t sa_hi = st + a32_bytes, sa_lo = sa_hi + a16_bytes;
                    const uint32_t sb_hi = sa_lo + a16_bytes, sb_lo = sb_hi + b_bytes;
#pragma unroll
                    for (int ks = 0; ks < kT2BK / 16; ++ks) {     // K = 16 per MMA: two 16-byte chunks
                        const uint64_t da_hi = umma_desc_kmajor(sa_hi + ks * 2 * lbo_a, lbo_a, sbo);
                        const uint64_t da_lo = umma_desc_kmajor(sa_lo + ks * 2 * lbo_a, lbo_a, sbo);
                        const uint64_t db_hi = umma_desc_kmajor(sb_hi + ks * 2 * lbo_b, lbo_b, sbo);
                        const uint64_t db_lo = umma_desc_kmajor(sb_lo + ks * 2 * lbo_b, lbo_b, sbo);
                        umma_f16(tmem_base, da_hi, db_hi, idesc, (kb | ks) != 0);             // hi . hi
                        umma_f16(tmem_base + acc_cols, da_hi, db_lo, idesc, (kb | ks) != 0);  // hi . lo
                        umma_f16(tmem_base + acc_cols, da_lo, db_hi, idesc, 1);               // lo . hi
                    }
                    umma_commit(&empty_bar[s]);                  // stage free once these MMAs have read it
                    if (kb == KB - 1) umma_commit(tmem_full);    // accumulators complete
                }
                __syncwarp();
                if (++s == stages) { s = 0; phase ^= 1; }
            }
            acc_phase ^= 1;
        }
    } else {
        // ===================== epilogue: warp w <-> TMEM lanes 32 (w % 4) .., column half w / 4 =====================
        uint32_t acc_phase = 0;
        const int lq = warp & 3, ch = warp >> 2;
        const int half_cols = (N_each / 2 + 15) / 16 * 16;     // columns per half, multiple of 16
        const int cbeg = ch * half_cols, cend = (ch + 1) * half_cols < N_each ? (ch + 1) * half_cols : N_each;
        const bool wide = (ldc & 7) == 0 && (reinterpret_cast<uintptr_t>(C) & 31) == 0;   // 32-byte aligned rows
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const long long mt = tile / n_nt;
            const int nt = (int)(tile - mt * n_nt);
            mbar_wait(tmem_full, acc_phase);
            tc_fence_after();
            const long long row = mt * kT2BM + lq * 32 + lane;
            float* crow = C + (size_t)(row < M ? row : 0) * ldc;
            const float rinv = tc_exp2(-tc_scale_exp(__int_as_float(__ldg(umax + row))));   // 2^-e_r
            const uint32_t lane_base = tmem_base + ((uint32_t)(lq * 32) << 16);
            for (int c0 = cbeg; c0 < cend; c0 += 32) {
                float v0[32], v1[32];
                tmem_ld32(lane_base + c0, v0);              // (reads past cend stay inside the allocated columns)
                tmem_ld32(lane_base + acc_cols + c0, v1);
                if (c0 + 32 >= cend) {   // this warp's last block is in registers: its share of the accumulators is free
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(tmem_empty);
                }
                if (row < M) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int cl = c0 + 8 * q;            // column inside the slice
                        const int c = nt * N_each + cl;       // gate column
                        // bias and colinv hold NP >= c + 8 entries
                        const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + c));
                        const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + c + 4));
                        const float4 f0 = __ldg(reinterpret_cast<const float4*>(colinv + c));
                        const float4 f1 = __ldg(reinterpret_cast<const float4*>(colinv + c + 4));
                        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                        const float ff[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
                        float o[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) o[e] = fmaf(v0[8 * q + e] + v1[8 * q + e], rinv * ff[e], bb[e]);
                        if (cl + 8 <= cend && c + 8 <= ldc && wide) {
                            asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n" ::"l"(crow + c),
                                         "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]), "f"(o[4]), "f"(o[5]), "f"(o[6]),
                                         "f"(o[7])
                                         : "memory");
                        } else {
#pragma unroll
                            for (int hq = 0; hq < 2; ++hq) {
                                const int c4 = c + 4 * hq;
                                if (cl + 4 * hq < cend && c4 < ldc)
                                    *reinterpret_cast<float4*>(crow + c4) =
                                        make_float4(o[4 * hq], o[4 * hq + 1], o[4 * hq + 2], o[4 * hq + 3]);
                            }
                        }
                    }
                }
            }
            acc_phase ^= 1;
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
