// GCN layers — relu((A_hat . X) . W + b), aggregate-then-transform, one or two layers fused.
//
// Reference: GraphConvLayer.forward, src/step5_gcn_layer_model.py:13-23 (matmul order :15,:18,
// ReLU :21); chained twice by GCN_GRU.forward, src/step6_gcn_gru_combined_model.py:17,20, whose
// `.view(1, T, S*13)` (:20) is the flat index s*F_out + f used for the output columns here.
//
// Work decomposition (dense A_hat, S small enough for A_hat^T to sit in shared memory):
//   * a CTA owns RB consecutive rows (a row = one (sequence, timestep) pair = an [S, F] slab).
//     The row block is contiguous in HBM in exactly the layout the kernel computes on, so it is
//     fetched with ONE bulk async copy (cp.async.bulk, the 1-D TMA path) completing on an
//     mbarrier; both layers then run in place in that buffer (aggregate -> barrier -> write);
//   * a thread owns SG consecutive stations of one row and keeps their aggregate in registers
//     as FEATURE pairs: the S-long aggregation is packed FP32 FMAs (FFMA2, sm_100a: two fp32
//     FMAs per instruction) acc2[s][fp] += (A[s][s'], A[s][s']) * (x[s'][2fp], x[s'][2fp+1]);
//     the F x F transform is FFMA2 too (pairs along the contracted feature index, two partial
//     sums added at the end);
//   * only the final slab goes to HBM: either row-major (single-layer op) or, for the fused
//     path, in the K-major 128-row tiles the input-projection GEMM copies with one bulk
//     async copy per stage (inproj.cuh), zero-padded to `ldo` columns.
#pragma once

#include "wg_common.cuh"

namespace wg {

constexpr int kGcnThreads = 128;
constexpr int kGcnUnroll = 2;      // aggregation loop unroll (measured: 1.88 -> 1.82 ms at S = 34)
constexpr int kGcnMinBlocks = 3;   // resident CTAs per SM the register budget is planned for (<= 168 regs)
constexpr int kGcnFS = 16;   // feature slots of the packed weight table
constexpr int kUTileRows = 128;  // rows per K-major tile of the tiled output (= inproj BM)

// floats of one row slab in shared memory: S stations x the widest feature dim of the layers
__host__ __device__ inline int gcn_row_stride(int S, int Fmax) { return S * Fmax; }

template <int FP, int SG>
__host__ __device__ inline size_t gcn_smem_floats(int S, int Fmax, int RB) {
    const int NSG = ceil_div(S, SG);
    size_t n = 0;
    n += (size_t)S * NSG * 8;           // adjT: [S][NSG][8] (SG <= 8 stations per group)
    n += 2 * (size_t)kGcnFS * kGcnFS;   // w1, w2: [f][fo] zero padded to 16 x 16
    n += 2 * (size_t)kGcnFS;            // b1, b2
    n += (size_t)round_up(RB * gcn_row_stride(S, Fmax), 4) + 4;  // slab block (+ mbarrier)
    return n;
}

// One GCN layer on the CTA's row block, in place in shared memory.
//   buf   [rows][RS]: a row holds [S][Fi] on entry and [S][Fo] on exit (RS >= S * max(Fi, Fo))
//   adjT  [S][NSG][8]: adjT[sp][q][i] = A_hat[q*SG+i][sp] (zero where out of range)
//   Wn    [16][16]: Wn[f][fo] = W[f][fo] (zero padded)
// Packed math (FFMA2 takes one operand as a scalar that it broadcasts to both halves):
//   aggregation  acc2[s][(f, f+1)]  += A[s][s']  * (x[s'][f], x[s'][f+1])
//   transform    o2[s][(fo, fo+1)]  += agg[s][f] * (W[f][fo], W[f][fo+1])
template <int FP, int SG, bool EXACT>
__device__ __noinline__ void gcn_layer_inplace(float* __restrict__ buf, const float* __restrict__ adjT,
                                               const float* __restrict__ Wn, const float* __restrict__ bias,
                                               int S, int Fi, int Fo, int RS, int NSG, int row_local, int q,
                                               bool active) {
    constexpr int FPP = (FP + 1) / 2;  // feature pairs
    float2 acc[SG][FPP];
    if (active) {
#pragma unroll
        for (int i = 0; i < SG; ++i)
#pragma unroll
            for (int fp = 0; fp < FPP; ++fp) acc[i][fp] = make_float2(0.0f, 0.0f);
        const float* xrow = buf + (size_t)row_local * RS;
        const float* arow = adjT + q * 8;
        const int astride = NSG * 8;
#pragma unroll kGcnUnroll
        for (int sp = 0; sp < S; ++sp) {
            float a[8];
            {
                const float4 t0 = *reinterpret_cast<const float4*>(arow + (size_t)sp * astride);
                a[0] = t0.x; a[1] = t0.y; a[2] = t0.z; a[3] = t0.w;
                if (SG > 4) {
                    const float4 t1 = *reinterpret_cast<const float4*>(arow + (size_t)sp * astride + 4);
                    a[4] = t1.x; a[5] = t1.y; a[6] = t1.z; a[7] = t1.w;
                }
            }
            float x[2 * FPP];
#pragma unroll
            for (int f = 0; f < 2 * FPP; ++f)
                x[f] = (f < FP && (EXACT || f < Fi)) ? xrow[sp * Fi + f] : 0.0f;
#pragma unroll
            for (int i = 0; i < SG; ++i) {
                const float2 aa = make_float2(a[i], a[i]);
#pragma unroll
                for (int fp = 0; fp < FPP; ++fp)
                    acc[i][fp] = __ffma2_rn(aa, make_float2(x[2 * fp], x[2 * fp + 1]), acc[i][fp]);
            }
        }
    }
    __syncthreads();  // every thread has finished reading the input slab
    if (active) {
        // transform: o2[s][(fo, fo+1)] += agg[s][f] (scalar operand, broadcast by FFMA2) * (W[f][fo], W[f][fo+1])
        float* orow = buf + (size_t)row_local * RS + q * SG * Fo;
#pragma unroll 1
        for (int fo0 = 0; fo0 < Fo; fo0 += 4) {
            float2 o[SG][2];
#pragma unroll
            for (int i = 0; i < SG; ++i) o[i][0] = o[i][1] = make_float2(0.0f, 0.0f);
            const bool second = fo0 + 2 < Fo;  // the chunk's upper fo pair exists
#pragma unroll
            for (int f = 0; f < FP; ++f) {
                const float4 w = *reinterpret_cast<const float4*>(Wn + f * kGcnFS + fo0);
#pragma unroll
                for (int i = 0; i < SG; ++i) {
                    const float av = (f & 1) ? acc[i][f >> 1].y : acc[i][f >> 1].x;
                    o[i][0] = __ffma2_rn(make_float2(av, av), make_float2(w.x, w.y), o[i][0]);
                    if (second) o[i][1] = __ffma2_rn(make_float2(av, av), make_float2(w.z, w.w), o[i][1]);
                }
            }
            const float4 bb = *reinterpret_cast<const float4*>(bias + fo0);
#pragma unroll
            for (int i = 0; i < SG; ++i) {
                if (q * SG + i < S) {
                    float* op = orow + i * Fo + fo0;
                    float u;
                    u = o[i][0].x + bb.x; op[0] = u < 0.0f ? 0.0f : u;  // ReLU; NaN propagates like torch.relu
                    if (fo0 + 1 < Fo) { u = o[i][0].y + bb.y; op[1] = u < 0.0f ? 0.0f : u; }
                    if (fo0 + 2 < Fo) { u = o[i][1].x + bb.z; op[2] = u < 0.0f ? 0.0f : u; }
                    if (fo0 + 3 < Fo) { u = o[i][1].y + bb.w; op[3] = u < 0.0f ? 0.0f : u; }
                }
            }
        }
    }
    __syncthreads();
}

// LAYERS == 2: GCN2(GCN1(x)) ; LAYERS == 1: GCN1(x) (W2/b2 unused, pass Fh = Fo = output width).
// TILED: out is [ceil(R/128)][ldo][128] (K-major row tiles, zero padded columns) else [R][ldo]
// row-major with ldo == S * F_last.
template <int FP, int SG, bool EXACT, int LAYERS, bool TILED>
__global__ void __launch_bounds__(kGcnThreads, kGcnMinBlocks)
    gcn_kernel(const float* __restrict__ X, const float* __restrict__ adj, const float* __restrict__ W1,
               const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2,
               float* __restrict__ out, long long R, int S, int Fi, int Fh, int Fo, int ldo, int RB) {
    extern __shared__ __align__(16) float smem[];
    const int NSG = ceil_div(S, SG);
    const int tid = threadIdx.x;
    const int Flast = LAYERS == 2 ? Fo : Fh;
    int Fmax = Fi > Fh ? Fi : Fh;
    if (LAYERS == 2 && Fo > Fmax) Fmax = Fo;
    const int RS = gcn_row_stride(S, Fmax);

    float* adjT = smem;
    float* w1d = adjT + (size_t)S * NSG * 8;
    float* w2d = w1d + kGcnFS * kGcnFS;
    float* b1s = w2d + kGcnFS * kGcnFS;
    float* b2s = b1s + kGcnFS;
    float* buf = b2s + kGcnFS;
    uint64_t* bar = reinterpret_cast<uint64_t*>(buf + round_up(RB * RS, 4));

    // ---- stage the (tiny) graph and layer parameters once per CTA ----
    for (int e = tid; e < S * NSG * 8; e += kGcnThreads) {
        const int sp = e / (NSG * 8);
        const int c = e % (NSG * 8);
        const int qq = c >> 3, i = c & 7;
        const int s = qq * SG + i;
        adjT[e] = (i < SG && s < S) ? adj[(size_t)s * S + sp] : 0.0f;
    }
    for (int e = tid; e < kGcnFS * kGcnFS; e += kGcnThreads) {
        const int f = e / kGcnFS, fo = e % kGcnFS;
        w1d[e] = (f < Fi && fo < Fh) ? W1[f * Fh + fo] : 0.0f;
        w2d[e] = (LAYERS == 2 && f < Fh && fo < Fo) ? W2[f * Fo + fo] : 0.0f;
    }
    for (int e = tid; e < kGcnFS; e += kGcnThreads) {
        b1s[e] = e < Fh ? b1[e] : 0.0f;
        b2s[e] = (LAYERS == 2 && e < Fo) ? b2[e] : 0.0f;
    }
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    __syncthreads();

    const int row_local = tid / NSG;
    const int q = tid % NSG;
    const long long nblocks = (R + RB - 1) / RB;
    const int in_cols = S * Fi;
    const int out_cols = S * Flast;
    // when the slab row is exactly one input row the block is one contiguous, TMA-copyable span
    const bool dense_rows = (RS == in_cols);
    unsigned phase = 0;

    for (long long rb = blockIdx.x; rb < nblocks; rb += gridDim.x) {
        const long long r0 = rb * RB;
        const int nrows = (int)((R - r0) < RB ? (R - r0) : RB);
        const float* src = X + (size_t)r0 * in_cols;
        const size_t bytes = (size_t)nrows * in_cols * 4;
        const bool bulk = dense_rows && ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && ((bytes & 15) == 0);
        if (bulk) {
            // ---- one bulk async copy of the whole row block, completion on the mbarrier ----
            if (tid == 0) {
                mbar_expect_tx(bar, (unsigned)bytes);
                bulk_g2s(buf, src, (unsigned)bytes, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1;
        } else {
            // ---- ragged / unaligned block: coalesced element copy ----
            const int n_in = nrows * in_cols;
            for (int e = tid; e < n_in; e += kGcnThreads) {
                const int row = e / in_cols;
                buf[row * RS + (e - row * in_cols)] = __ldg(src + e);
            }
            __syncthreads();
        }

        const bool active = row_local < nrows;
        gcn_layer_inplace<FP, SG, EXACT>(buf, adjT, w1d, b1s, S, Fi, Fh, RS, NSG, row_local, q, active);
        if (LAYERS == 2)
            gcn_layer_inplace<FP, SG, EXACT>(buf, adjT, w2d, b2s, S, Fh, Fo, RS, NSG, row_local, q, active);

        // ---- store the final slab ----
        if (TILED) {
            // out[(r / 128)][c][r % 128]: a lane owns one row of the block (its tile offset is fixed),
            // each warp walks the columns; a store instruction writes nrows consecutive floats
            for (int rl = tid & 31; rl < nrows; rl += 32) {
                const long long r = r0 + rl;
                float* dstc = out + (size_t)(r / kUTileRows) * ldo * kUTileRows + (r % kUTileRows);
                const float* srcr = buf + rl * RS;
                for (int c = tid >> 5; c < ldo; c += kGcnThreads / 32)
                    dstc[(size_t)c * kUTileRows] = c < out_cols ? srcr[c] : 0.0f;
            }
        } else {
            float* dst = out + (size_t)r0 * ldo;
            const int n_out = nrows * ldo;
            for (int e = tid; e < n_out; e += kGcnThreads) {
                const int row = e / ldo;
                dst[e] = buf[row * RS + (e - row * ldo)];
            }
        }
        __syncthreads();  // the slab is free again (generic reads done before the next async write)
    }
}

}  // namespace wg
