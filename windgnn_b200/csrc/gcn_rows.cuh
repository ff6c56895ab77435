// Both GCN layers of the 13-feature model, second generation: lane = row, warp = station group.
//
// Reference: GraphConvLayer.forward, src/step5_gcn_layer_model.py:13-23 (matmul order :15,:18,
// ReLU :21), chained twice by GCN_GRU.forward, src/step6_gcn_gru_combined_model.py:17,20; the
// `.view(1, T, S*13)` of :20 is the flat column index s*13 + f of the output.
//
// gcn_kernel (gcn.cuh) maps a thread to (row, 7 stations): the final slab has to go back through
// shared memory to reach the K-major tiles of the projection GEMM (a 96-byte run per store
// instruction, ~670 instructions per thread and block), 8 of 128 lanes idle, and 53 % of the issued
// instructions are not FMAs (ncu r01: FMA pipe 60 %).  Here
//   * a CTA owns 32 consecutive rows (a row = one (sequence, timestep) pair = an [S, 13] slab),
//     LANE = row; a warp owns a group of station PAIRS for all 32 rows;
//   * aggregation  acc2[(s, s+1)][f] += x[s'][f] * (A[s][s'], A[s+1][s'])  — FFMA2 with the feature
//     value as the broadcast scalar and the adjacency pair warp-uniform (one broadcast LDS.128 per
//     four stations); exactly 13 features, no padded feature lane;
//   * transform    o2[(s, s+1)][fo] += W[f][fo] * acc2[(s, s+1)][f]  — the accumulator pair IS the
//     operand pair; the weight is a warp-uniform scalar;
//   * layer 1 writes its result back to shared memory in a padded [row][station][16] layout
//     (16-byte loads for layer 2, row stride = 4 mod 32 floats: conflict free);
//   * layer 2's result goes from registers straight to the K-major tiles of the projection GEMM:
//     for a fixed column the 32 lanes are 32 consecutive rows, i.e. one 128-byte store.
// The input block arrives with ONE bulk async copy (cp.async.bulk), as before.
//
// Every sum runs in the order of gcn_kernel (s' ascending, then f ascending, bias added last), so the
// two kernels are bit-identical (tested); this one serves F_in = F_hid = F_out = 13 (the only widths
// the reference's forward accepts: the 13 is hard-coded at step6:16) and S <= 48.
#pragma once

#include "gcn.cuh"
#include "wg_common.cuh"

namespace wg {

constexpr int kGrRows = 32;     // rows per block (= lanes)
constexpr int kGrF = 13;        // feature width served
constexpr int kGrFS = 16;       // feature stride of the layer-1 result in shared memory
constexpr int kGrAP = 12;       // adjacency floats per (s', warp): up to 6 station pairs
constexpr int kGrMaxPairs = 5;  // station pairs per warp (accumulators: 5 x 13 float2 = 130 registers)
constexpr int kGrMaxWarps = 8;

__host__ __device__ inline int gcn_rows_warps(int S) { return ceil_div(ceil_div(S, 2), kGrMaxPairs); }
__host__ __device__ inline bool gcn_rows_applies(int S, int Fi, int Fh, int Fo) {
    return Fi == kGrF && Fh == kGrF && Fo == kGrF && gcn_rows_warps(S) <= kGrMaxWarps && S <= 48;
}
__host__ __device__ inline int gcn_rows_rs2(int S) { return S * kGrFS + 4; }
// Balanced mode (17 station pairs over 4 warps, i.e. S = 33 / 34): every warp owns 4 pairs and the 17th pair is
// SHARED — warp w aggregates it for the feature slice 3w .. 3w + 3 and, after the barrier that follows the
// aggregation anyway, transforms it for the same slice of output columns; the aggregate travels through a
// [32 rows][28] exchange buffer per layer.  Every sum keeps its order (s' ascending, f ascending), so the result
// is bit-identical to the 5/4/4/4 split, whose light warps spent 20 % of their time at the CTA barriers
// (ncu: 16 % of all warp samples) waiting for the warp with five pairs.
constexpr int kGrXS = 28;   // exchange row stride (floats): 13 float2, padded; 8 lanes x 16 B cover all 32 banks
__host__ __device__ inline bool gcn_rows_balanced(int S) { return ceil_div(S, 2) == 17; }
// warp w's slice: features / output columns 3w .. 3w + 3 (0-3, 3-6, 6-9, 9-12; the boundary columns are computed
// by two warps — the same value, stored twice — so that all four warps run ONE instruction stream: with a slice per
// template instantiation the four warps of a CTA executed four copies of the block code and the kernel ran at
// half speed on instruction-cache misses)
constexpr int kGrSliceStep = 3;
constexpr int kGrSliceW = 4;
__host__ __device__ inline size_t gcn_rows_smem_floats(int S) {
    const int NW = gcn_rows_warps(S);
    size_t n = (size_t)S * NW * kGrAP;                 // adjW[s'][warp][12]
    n += 2 * (size_t)kGcnFS * kGcnFS + 2 * kGcnFS;     // w1, w2, b1, b2 (zero padded 16 x 16 / 16)
    const size_t in_f = (size_t)kGrRows * S * kGrF, g1_f = (size_t)kGrRows * gcn_rows_rs2(S);
    n += round_up((int)(in_f > g1_f ? in_f : g1_f), 4) + 4;   // slab block (+ mbarrier)
    if (gcn_rows_balanced(S)) n += 2 * (size_t)kGrRows * kGrXS;   // shared-pair exchange, one buffer per layer
    return n;
}

// acc[p][f] = sum_{s'} x[s'][f] * (A[2p][s'], A[2p+1][s'])  for this warp's NPW station pairs.
// PADDED: x row is [S][16] (layer-1 result) else [S][13] as it sits in HBM (VEC: the row length S*13 is
// even, so every row base is 8-byte aligned and the loads are 8 bytes wide where the offset is even).
// The operands of step s'+1 are loaded BEFORE the FMAs of step s' are issued (two register fragments): with two
// warps per scheduler the ~30 cycles from LDS to the first dependent FFMA2 were exposed once per step (ncu:
// 11 % of the samples waiting on shared-memory data).  VEC is a template parameter so that the loop body has no
// branch (the r02 body branched on it, which kept the loads of a step behind the FMAs of the previous one).
// SHARED: balanced mode, this warp's slice of the shared pair (its adjacency pair sits behind the NPW own pairs;
// the slice's four x values are loaded separately at the runtime offset f0 — the register copy of the row cannot
// be indexed at run time)
template <int NPW, bool SHARED>
struct GrFrag {
    static constexpr int NA4 = (NPW + (SHARED ? 1 : 0) + 1) / 2;   // float4 loads of adjacency values
    float a[NA4 * 4];
    float x[kGrF];
    float xs[kGrSliceW];
};

template <int NPW, bool PADDED, bool VEC, bool SHARED>
__device__ __forceinline__ void gr_aggregate_x(float2 (&acc)[NPW][kGrF], float2 (&accs)[4],
                                               const float* __restrict__ xrow, const float* __restrict__ arow,
                                               int astride, int S, int fs0) {
    using Frag = GrFrag<NPW, SHARED>;
#pragma unroll
    for (int j = 0; j < 4; ++j) accs[j] = make_float2(0.0f, 0.0f);
#pragma unroll
    for (int p = 0; p < NPW; ++p)
#pragma unroll
        for (int f = 0; f < kGrF; ++f) acc[p][f] = make_float2(0.0f, 0.0f);
    auto load = [&](Frag& fr, int sp, auto odd_tag) {
        constexpr bool ODD = decltype(odd_tag)::value != 0;
        const float* ap = arow + (size_t)sp * astride;
#pragma unroll
        for (int q = 0; q < Frag::NA4; ++q) {
            const float4 t = *reinterpret_cast<const float4*>(ap + 4 * q);
            fr.a[4 * q] = t.x; fr.a[4 * q + 1] = t.y; fr.a[4 * q + 2] = t.z; fr.a[4 * q + 3] = t.w;
        }
        if constexpr (SHARED) {
            const float* xq = xrow + sp * (PADDED ? kGrFS : kGrF) + fs0;
#pragma unroll
            for (int j = 0; j < kGrSliceW; ++j) fr.xs[j] = xq[j];
        }
        if (PADDED) {
            const float* xp = xrow + sp * kGrFS;
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const float4 t = *reinterpret_cast<const float4*>(xp + 4 * q);
                fr.x[4 * q] = t.x; fr.x[4 * q + 1] = t.y; fr.x[4 * q + 2] = t.z; fr.x[4 * q + 3] = t.w;
            }
            fr.x[12] = xp[12];
        } else {
            const float* xp = xrow + sp * kGrF;
            if (!VEC) {   // odd row length (odd S): the rows are only 4-byte aligned
#pragma unroll
                for (int f = 0; f < kGrF; ++f) fr.x[f] = xp[f];
            } else if (!ODD) {   // even offset: pairs (0,1) .. (10,11), then 12
#pragma unroll
                for (int q = 0; q < 6; ++q) {
                    const float2 t = *reinterpret_cast<const float2*>(xp + 2 * q);
                    fr.x[2 * q] = t.x; fr.x[2 * q + 1] = t.y;
                }
                fr.x[12] = xp[12];
            } else {      // odd offset: 0, then pairs (1,2) .. (11,12)
                fr.x[0] = xp[0];
#pragma unroll
                for (int q = 0; q < 6; ++q) {
                    const float2 t = *reinterpret_cast<const float2*>(xp + 1 + 2 * q);
                    fr.x[1 + 2 * q] = t.x; fr.x[2 + 2 * q] = t.y;
                }
            }
        }
    };
    auto fma = [&](const Frag& fr) {
#pragma unroll
        for (int p = 0; p < NPW; ++p) {
            const float2 aa = make_float2(fr.a[2 * p], fr.a[2 * p + 1]);
#pragma unroll
            for (int f = 0; f < kGrF; ++f) acc[p][f] = __ffma2_rn(make_float2(fr.x[f], fr.x[f]), aa, acc[p][f]);
        }
        if constexpr (SHARED) {
            const float2 aa = make_float2(fr.a[2 * NPW], fr.a[2 * NPW + 1]);
#pragma unroll
            for (int j = 0; j < kGrSliceW; ++j) accs[j] = __ffma2_rn(make_float2(fr.xs[j], fr.xs[j]), aa, accs[j]);
        }
    };
    // s' ascending, as before (the sums are bit-identical to gcn_kernel's)
    Frag f0, f1;
    load(f0, 0, IntC<0>{});
    int sp = 0;
#pragma unroll 1
    for (; sp + 2 < S; sp += 2) {
        load(f1, sp + 1, IntC<1>{});
        fma(f0);
        load(f0, sp + 2, IntC<0>{});
        fma(f1);
    }
    if (sp + 1 < S) {
        load(f1, sp + 1, IntC<1>{});
        fma(f0);
        fma(f1);
    } else {
        fma(f0);
    }
}

template <int NPW, bool PADDED, bool VEC>
__device__ __forceinline__ void gr_aggregate(float2 (&acc)[NPW][kGrF], const float* __restrict__ xrow,
                                             const float* __restrict__ arow, int astride, int S) {
    float2 unused[4];
    gr_aggregate_x<NPW, PADDED, VEC, false>(acc, unused, xrow, arow, astride, S, 0);
}

// The shared pair's transform for this warp's slice of output columns: o[j] = sum_f W[f][c0 + j] * agg[f]
// (f ascending), agg = the pair's 13 aggregated features of this lane's row, read back from the exchange row.
__device__ __forceinline__ void gr_transform_shared(float2 (&o)[kGrSliceW], const float* __restrict__ xrow,
                                                    const float* __restrict__ Wn, int c0) {
    float2 agg[kGrF + 1];
#pragma unroll
    for (int q = 0; q < 7; ++q) {
        const float4 t = *reinterpret_cast<const float4*>(xrow + 4 * q);
        agg[2 * q] = make_float2(t.x, t.y);
        agg[2 * q + 1] = make_float2(t.z, t.w);
    }
#pragma unroll
    for (int j = 0; j < kGrSliceW; ++j) o[j] = make_float2(0.0f, 0.0f);
    const float* wp = Wn + c0;
#pragma unroll
    for (int f = 0; f < kGrF; ++f)
#pragma unroll
        for (int j = 0; j < kGrSliceW; ++j) {
            const float wv = wp[f * kGcnFS + j];
            o[j] = __ffma2_rn(make_float2(wv, wv), agg[f], o[j]);
        }
}

// o[p][c] = sum_f W[f][c0 + c] * acc[p][f]  for one chunk of WIDTH output features (f ascending)
template <int NPW, int WIDTH>
__device__ __forceinline__ void gr_transform_chunk(float2 (&o)[NPW][4], const float2 (&acc)[NPW][kGrF],
                                                   const float* __restrict__ Wn, int c0) {
#pragma unroll
    for (int p = 0; p < NPW; ++p)
#pragma unroll
        for (int c = 0; c < 4; ++c) o[p][c] = make_float2(0.0f, 0.0f);
#pragma unroll
    for (int f = 0; f < kGrF; ++f) {
        const float4 w = *reinterpret_cast<const float4*>(Wn + f * kGcnFS + c0);
        const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int p = 0; p < NPW; ++p)
#pragma unroll
            for (int c = 0; c < WIDTH; ++c) o[p][c] = __ffma2_rn(make_float2(wv[c], wv[c]), acc[p][f], o[p][c]);
    }
}

// ReLU; NaN propagates like torch.relu.  One FMNMX.NAN instead of FSETP + FSEL (the epilogues run 884 of these per
// row).
__device__ __forceinline__ float gr_relu(float u) {
    float r;
    asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(r) : "f"(u));
    return r;
}
// (o.x + b, o.y + b): one FADD2 for the two stations of a pair
__device__ __forceinline__ float2 gr_bias(float2 o, float b) { return __fadd2_rn(o, make_float2(b, b)); }

// One row block through both layers for a warp that owns NPW station pairs starting at station s0.
// SHARED (balanced mode): additionally this warp's feature / column slice f0 .. f0 + 3 of the shared pair
// (stations 32, 33); xch = this lane's two exchange rows (layer 1, layer 2: kGrRows * kGrXS floats apart).
// ROWMAX (tensor path): the largest value this warp writes to the lane's row goes to *umax_row (atomicMax of the
// float bits, which order like integers for U >= 0).
template <int NPW, bool SHARED, bool ROWMAX>
__device__ __forceinline__ void gr_block(float* __restrict__ buf, const float* __restrict__ arow, int astride,
                                         const float* __restrict__ w1d, const float* __restrict__ b1s,
                                         const float* __restrict__ w2d, const float* __restrict__ b2s, int S, int s0,
                                         int lane, bool row_ok, float* __restrict__ out_col0, int ldo, bool pad_warp,
                                         const float* __restrict__ next_src, unsigned next_bytes, uint64_t* bar,
                                         float* __restrict__ xch, int f0, int* __restrict__ umax_row) {
    constexpr int SNF = kGrSliceW;
    constexpr int SS = 32;   // the shared pair's first station (pair 16)
    const int SF0 = f0;
    const int in_cols = S * kGrF, RS2 = gcn_rows_rs2(S);
    float2 acc[NPW][kGrF];
    float2 accs[4];
    auto put_shared = [&](float* row) {   // this warp's slice of the shared pair's aggregate -> exchange row
#pragma unroll
        for (int j = 0; j < SNF; ++j) *reinterpret_cast<float2*>(row + 2 * (SF0 + j)) = accs[j];
    };
    // ---- layer 1 ----
    if ((in_cols & 1) == 0)
        gr_aggregate_x<NPW, false, true, SHARED>(acc, accs, buf + (size_t)lane * in_cols, arow, astride, S, f0);
    else
        gr_aggregate_x<NPW, false, false, SHARED>(acc, accs, buf + (size_t)lane * in_cols, arow, astride, S, f0);
    if (SHARED) put_shared(xch);
    __syncthreads();   // every warp has finished reading the input slab: the padded layer-1 result may overwrite it
    float* g1row = buf + (size_t)lane * RS2;
    auto store_g1 = [&](const float2 (&o)[NPW][4], int c0) {
        const float4 bb = *reinterpret_cast<const float4*>(b1s + c0);
        const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
        for (int p = 0; p < NPW; ++p) {
            const int s = s0 + 2 * p;
            float4 v0, v1;   // columns >= 13 come out as relu(0 + 0) = 0: the padding is defined
            const float2 u0 = gr_bias(o[p][0], bv[0]), u1 = gr_bias(o[p][1], bv[1]);
            const float2 u2 = gr_bias(o[p][2], bv[2]), u3 = gr_bias(o[p][3], bv[3]);
            v0.x = gr_relu(u0.x); v0.y = gr_relu(u1.x); v0.z = gr_relu(u2.x); v0.w = gr_relu(u3.x);
            v1.x = gr_relu(u0.y); v1.y = gr_relu(u1.y); v1.z = gr_relu(u2.y); v1.w = gr_relu(u3.y);
            *reinterpret_cast<float4*>(g1row + s * kGrFS + c0) = v0;   // s < S for every owned pair (pairs < ceil(S/2))
            if (s + 1 < S) *reinterpret_cast<float4*>(g1row + (s + 1) * kGrFS + c0) = v1;
        }
    };
    {
        float2 o[NPW][4];
#pragma unroll 1
        for (int c0 = 0; c0 < 12; c0 += 4) {   // output features 0 .. 11
            gr_transform_chunk<NPW, 4>(o, acc, w1d, c0);
            store_g1(o, c0);
        }
        gr_transform_chunk<NPW, 1>(o, acc, w1d, 12);   // feature 12 (kGrF == 13)
        store_g1(o, 12);
    }
    if (SHARED) {   // shared pair, this warp's output columns SF0 .. SF0 + SNF - 1
        float2 o[4];
        gr_transform_shared(o, xch, w1d, SF0);
#pragma unroll
        for (int j = 0; j < SNF; ++j) {
            const float2 u = gr_bias(o[j], b1s[SF0 + j]);
            g1row[SS * kGrFS + SF0 + j] = gr_relu(u.x);
            if (SS + 1 < S) g1row[(SS + 1) * kGrFS + SF0 + j] = gr_relu(u.y);
        }
    }
    __syncthreads();   // layer-1 result complete
    // ---- layer 2 ----
    gr_aggregate_x<NPW, true, true, SHARED>(acc, accs, g1row, arow, astride, S, f0);
    if (SHARED) put_shared(xch + kGrRows * kGrXS);
    __syncthreads();   // the slab is free: every warp holds its layer-2 aggregate in registers
    // the next block's bulk copy starts NOW and lands while this block's transform / stores run from registers
    if (next_bytes != 0 && threadIdx.x == 0) {
        mbar_expect_tx(bar, next_bytes);
        bulk_g2s(buf, next_src, next_bytes, bar);
    }
    float vmax = 0.0f;   // ROWMAX
    auto store_u = [&](const float2 (&o)[NPW][4], int c0, auto width) {
        constexpr int W = decltype(width)::value;
        const float4 bb = *reinterpret_cast<const float4*>(b2s + c0);
        const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
        if (row_ok) {
#pragma unroll
            for (int p = 0; p < NPW; ++p) {
                const int s = s0 + 2 * p;
                // column s*13 + fo of the tile: 128 floats per column, this lane's row inside it
                float* c_lo = out_col0 + (size_t)(s * kGrF + c0) * kUTileRows;
#pragma unroll
                for (int c = 0; c < W; ++c) {
                    const float2 u = gr_bias(o[p][c], bv[c]);
                    c_lo[(size_t)c * kUTileRows] = gr_relu(u.x);
                    if (s + 1 < S) c_lo[(size_t)(kGrF + c) * kUTileRows] = gr_relu(u.y);
                    if (ROWMAX) vmax = fmaxf(vmax, s + 1 < S ? fmaxf(gr_relu(u.x), gr_relu(u.y)) : gr_relu(u.x));
                }
            }
        }
    };
    {
        float2 o[NPW][4];
#pragma unroll 1
        for (int c0 = 0; c0 < 12; c0 += 4) {
            gr_transform_chunk<NPW, 4>(o, acc, w2d, c0);
            store_u(o, c0, IntC<4>{});
        }
        gr_transform_chunk<NPW, 1>(o, acc, w2d, 12);
        store_u(o, 12, IntC<1>{});
    }
    if (SHARED) {
        float2 o[4];
        gr_transform_shared(o, xch + kGrRows * kGrXS, w2d, SF0);
        if (row_ok) {
            float* c_lo = out_col0 + (size_t)(SS * kGrF + SF0) * kUTileRows;
#pragma unroll
            for (int j = 0; j < SNF; ++j) {
                const float2 u = gr_bias(o[j], b2s[SF0 + j]);
                c_lo[(size_t)j * kUTileRows] = gr_relu(u.x);
                if (SS + 1 < S) c_lo[(size_t)(kGrF + j) * kUTileRows] = gr_relu(u.y);
                if (ROWMAX) vmax = fmaxf(vmax, SS + 1 < S ? fmaxf(gr_relu(u.x), gr_relu(u.y)) : gr_relu(u.x));
            }
        }
    }
    if (pad_warp && row_ok)   // zero the K padding of the projection GEMM
        for (int c = in_cols; c < ldo; ++c) out_col0[(size_t)c * kUTileRows] = 0.0f;
    if (ROWMAX && row_ok) atomicMax(umax_row, __float_as_int(vmax));
}

// X [R][S][13] -> out [ceil(R/128)][ldo][128] (K-major row tiles, columns >= S*13 zero)
// ROWMAX (the tensor path's instantiation): also umax[r] = max(umax[r], the largest element of U row r), float bits
// (umax cleared by the caller)
template <bool ROWMAX>
__global__ void __launch_bounds__(kGrMaxWarps * 32, 1)
    gcn_rows_kernel(const float* __restrict__ X, const float* __restrict__ adj, const float* __restrict__ W1,
                    const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2,
                    float* __restrict__ out, long long R, int S, int ldo, int* __restrict__ umax) {
    extern __shared__ __align__(16) float smem[];
    const int NW = gcn_rows_warps(S);
    const int nthreads = NW * 32;
    const int tid = threadIdx.x, lane = tid & 31;
    const int in_cols = S * kGrF;
    // station pairs are dealt out as evenly as possible; the warps with one more pair are rotated
    // with the CTA's wave so that co-resident CTAs do not put their heavy warps on one scheduler
    // (balanced mode: four pairs per warp, the 17th is shared by feature slice — no heavy warp)
    const bool balanced = gcn_rows_balanced(S);
    const int NPT = balanced ? 16 : ceil_div(S, 2), base = NPT / NW, extra = NPT % NW;
    const int w = ((tid >> 5) + (blockIdx.x / kNumSMs) * 2) % NW;
    const int npw = base + (w < extra ? 1 : 0);
    const int p0 = w * base + (w < extra ? w : extra);
    const int s0 = 2 * p0;

    float* adjW = smem;                                   // [S][NW][12]
    float* w1d = adjW + (size_t)S * NW * kGrAP;
    float* w2d = w1d + kGcnFS * kGcnFS;
    float* b1s = w2d + kGcnFS * kGcnFS;
    float* b2s = b1s + kGcnFS;
    float* buf = b2s + kGcnFS;
    const size_t in_f = (size_t)kGrRows * in_cols, g1_f = (size_t)kGrRows * gcn_rows_rs2(S);
    uint64_t* bar = reinterpret_cast<uint64_t*>(buf + round_up((int)(in_f > g1_f ? in_f : g1_f), 4));
    float* xch = reinterpret_cast<float*>(bar) + 4 + (size_t)lane * kGrXS;   // balanced mode: [2][32][28] after the mbarrier

    for (int e = tid; e < S * NW * kGrAP; e += nthreads) {
        const int sp = e / (NW * kGrAP), c = e % (NW * kGrAP);
        const int ww = c / kGrAP, i = c % kGrAP;
        const int wn = base + (ww < extra ? 1 : 0), ws0 = 2 * (ww * base + (ww < extra ? ww : extra));
        // balanced mode: the shared pair's adjacency values follow the warp's own pairs in every warp's slot
        const int s = i < 2 * wn ? ws0 + i : (balanced && i < 2 * wn + 2 ? 32 + (i - 2 * wn) : S);
        adjW[e] = s < S ? adj[(size_t)s * S + sp] : 0.0f;
    }
    for (int e = tid; e < kGcnFS * kGcnFS; e += nthreads) {
        const int f = e / kGcnFS, fo = e % kGcnFS;
        const bool in = f < kGrF && fo < kGrF;
        w1d[e] = in ? W1[f * kGrF + fo] : 0.0f;
        w2d[e] = in ? W2[f * kGrF + fo] : 0.0f;
    }
    for (int e = tid; e < kGcnFS; e += nthreads) {
        b1s[e] = e < kGrF ? b1[e] : 0.0f;
        b2s[e] = e < kGrF ? b2[e] : 0.0f;
    }
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    __syncthreads();

    const float* arow = adjW + w * kGrAP;
    const int astride = NW * kGrAP;
    const long long nblocks = (R + kGrRows - 1) / kGrRows;
    unsigned phase = 0;
    // a block is bulk-copyable when its span is 16-byte aligned and a 16-byte multiple
    auto block_span = [&](long long rb, const float*& src, unsigned& bytes, int& nrows) {
        const long long r0 = rb * kGrRows;
        nrows = (int)((R - r0) < kGrRows ? (R - r0) : kGrRows);
        src = X + (size_t)r0 * in_cols;
        bytes = (unsigned)((size_t)nrows * in_cols * 4);
        return ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && ((bytes & 15) == 0);
    };
    bool prefetched = false;   // the current block's bulk copy was issued during the previous block
    for (long long rb = blockIdx.x; rb < nblocks; rb += gridDim.x) {
        const long long r0 = rb * kGrRows;
        const float* src;
        unsigned bytes;
        int nrows;
        const bool bulk = block_span(rb, src, bytes, nrows);
        if (bulk) {
            if (!prefetched && tid == 0) {
                mbar_expect_tx(bar, bytes);
                bulk_g2s(buf, src, bytes, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1;
        } else {   // ragged / unaligned block: coalesced element copy
            const int n_in = nrows * in_cols;
            for (int e = tid; e < n_in; e += nthreads) buf[e] = __ldg(src + e);
            __syncthreads();
        }
        // the block after this one (same CTA): prefetched from inside gr_block when bulk-copyable
        const float* nsrc = nullptr;
        unsigned nbytes = 0;
        int nn;
        prefetched = false;
        if (rb + gridDim.x < nblocks && block_span(rb + gridDim.x, nsrc, nbytes, nn)) prefetched = true;
        else nbytes = 0;
        const long long r = r0 + lane;
        float* out_col0 = out + (size_t)(r / kUTileRows) * ldo * kUTileRows + (r % kUTileRows);
        const bool row_ok = lane < nrows;
        const bool pad_warp = w == NW - 1;
        int* umax_row = ROWMAX ? umax + r : nullptr;
#define WG_GR(N)                                                                                              \
    case N:                                                                                                   \
        gr_block<N, false, ROWMAX>(buf, arow, astride, w1d, b1s, w2d, b2s, S, s0, lane, row_ok, out_col0, ldo, \
                                   pad_warp, nsrc, nbytes, bar, xch, 0, umax_row);                            \
        break;
        if (balanced) {   // one instruction stream for the four warps; the slice offset is a runtime value
            gr_block<4, true, ROWMAX>(buf, arow, astride, w1d, b1s, w2d, b2s, S, s0, lane, row_ok, out_col0, ldo,
                                      pad_warp, nsrc, nbytes, bar, xch, kGrSliceStep * w, umax_row);
        } else {
            switch (npw) {   // warp-uniform
                WG_GR(1) WG_GR(2) WG_GR(3) WG_GR(4) WG_GR(5)
                default: break;
            }
        }
#undef WG_GR
        // gr_block's last barrier separates this block's reads of the slab from the next bulk copy
    }
}

}  // namespace wg
