// Backward of the two fused GCN layers — weight and bias gradients from dL/dU.
//
// Reference: autograd through GraphConvLayer.forward (src/step5_gcn_layer_model.py:13-23) applied
// twice (src/step6_gcn_gru_combined_model.py:17,20).  Per (sequence, timestep) row, with
//   AX = A.X    G1 = relu(AX.W1 + b1)    AG = A.G1    U = relu(AG.W2 + b2):
//   dZ2 = dU * [AG.W2 + b2 > 0]     dW2 += AG^T dZ2     db2 += colsum(dZ2)
//   dAG = dZ2 W2^T                  dG1 = A^T dAG       dZ1 = dG1 * [G1 > 0]
//   dW1 += AX^T dZ1                 db1 += colsum(dZ1)
// (no gradient is needed for X or for the adjacency — both are data).  Nothing of the forward's
// GCN stage is saved: AX, G1, AG are recomputed from X here (they are 2 x 13 KB per row of
// intermediate state that would otherwise go through HBM).
//
// Same decomposition as the forward kernel (gcn.cuh): a CTA owns RB rows, the X and dU row
// blocks arrive by ONE bulk async copy each, a thread owns kGbwSG = 4 stations of one row and does the
// S-long aggregations with FFMA2 on feature pairs.  The slabs live in shared memory with 16
// floats per station so that the two 13 x 13 outer-product reductions (sum over all stations of
// all rows of the block) run as a small register-tiled GEMM: thread = 4 x 4 output tile x one of
// 8 slices of the (row, station) index, operands by LDS.128.  Those accumulators persist in
// registers across the CTA's row blocks; per-thread partials go to HBM once, and
// gcn_bwd_finish_kernel adds them in a fixed order (deterministic).
#pragma once

#include "gcn.cuh"
#include "wg_common.cuh"

namespace wg {

constexpr int kGbwW = 16;   // width of the zero-padded weight tables
constexpr int kGbwFS = 20;  // floats per station in the padded slabs: 16 used + 4 so that the stations a warp's
                            // lanes own (consecutive stations, 80 B apart) fall into distinct bank groups
constexpr int kGbwThreads = 256;
// stations per thread: the slabs bound the CTA to ~24 rows, so the narrower station group is what puts 7 warps
// instead of 4 on the SM
constexpr int kGbwSG = 4;
// padded slab row stride: + 4 floats so that the rows a warp touches at once start in different banks
__host__ __device__ inline int gcn_bwd_row_stride(int S) { return S * kGbwFS + 4; }

// The adjacency tables keep 8 floats per (station, group) although the kernel reads 4: this size decides the row
// block RB, and RB the grouping of the partial sums, so the gradient bits depend on it.
__host__ __device__ inline size_t gcn_bwd_smem_floats(int S, int ldu, int RB) {
    const int NSG = ceil_div(S, kGbwSG);
    size_t n = 0;
    n += 2 * (size_t)S * NSG * 8;          // adjT (A[own][sp]) and adjN (A[sp][own])
    n += 3 * (size_t)kGbwW * kGbwW;        // W1, W2, W2^T (zero padded 16 x 16)
    n += 2 * (size_t)kGbwW;                // b1, b2
    n += 3 * (size_t)RB * gcn_bwd_row_stride(S);  // padded slabs s0, s1, s2
    n += (size_t)round_up(RB * ldu, 4);    // dU block (row stride ldu >= S * F_out)
    n += 4;                                // mbarrier
    return n;
}

// acc[i][fp] = sum_sp tab[sp][q][i] * (x[sp][2fp], x[sp][2fp+1]); x rows `stride` floats apart,
// features >= flim read as zero (dense input slab) or are zero padding (stride 16 slabs).
// VEC: the slab is a padded one (16 floats per station, 16-byte aligned): features come by LDS.128.
template <int FPP, bool VEC>
__device__ __forceinline__ void gcn_bwd_agg(float2 (&acc)[kGbwSG][FPP], const float* __restrict__ xrow, int stride,
                                            int flim, const float* __restrict__ arow, int astride, int S) {
#pragma unroll
    for (int i = 0; i < kGbwSG; ++i)
#pragma unroll
        for (int fp = 0; fp < FPP; ++fp) acc[i][fp] = make_float2(0.0f, 0.0f);
#pragma unroll 2
    for (int sp = 0; sp < S; ++sp) {
        const float4 t = *reinterpret_cast<const float4*>(arow + (size_t)sp * astride);
        const float a[kGbwSG] = {t.x, t.y, t.z, t.w};
        float x[2 * FPP + 2];
        if (VEC) {
#pragma unroll
            for (int v = 0; v < (2 * FPP + 3) / 4; ++v) {
                const float4 t = *reinterpret_cast<const float4*>(xrow + sp * kGbwFS + 4 * v);
                x[4 * v] = t.x;
                x[4 * v + 1] = t.y;
                if (4 * v + 2 < 2 * FPP) { x[4 * v + 2] = t.z; x[4 * v + 3] = t.w; }
            }
        } else {
#pragma unroll
            for (int f = 0; f < 2 * FPP; ++f) x[f] = f < flim ? xrow[sp * stride + f] : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < kGbwSG; ++i) {
            const float2 aa = make_float2(a[i], a[i]);
#pragma unroll
            for (int fp = 0; fp < FPP; ++fp)
                acc[i][fp] = __ffma2_rn(aa, make_float2(x[2 * fp], x[2 * fp + 1]), acc[i][fp]);
        }
    }
}

// o[i][0..1] = sum_f in[i][f] * (W[f][fo0 .. fo0+3]) for this thread's kGbwSG stations
template <int FPP>
__device__ __forceinline__ void gcn_bwd_xform4(float2 (&o)[kGbwSG][2], const float2 (&in)[kGbwSG][FPP],
                                               const float* __restrict__ Wn, int fo0) {
#pragma unroll
    for (int i = 0; i < kGbwSG; ++i) o[i][0] = o[i][1] = make_float2(0.0f, 0.0f);
#pragma unroll
    for (int f = 0; f < 2 * FPP; ++f) {
        const float4 w = *reinterpret_cast<const float4*>(Wn + f * kGbwW + fo0);
#pragma unroll
        for (int i = 0; i < kGbwSG; ++i) {
            const float av = (f & 1) ? in[i][f >> 1].y : in[i][f >> 1].x;
            o[i][0] = __ffma2_rn(make_float2(av, av), make_float2(w.x, w.y), o[i][0]);
            o[i][1] = __ffma2_rn(make_float2(av, av), make_float2(w.z, w.w), o[i][1]);
        }
    }
}

// FP: compile-time bound on the feature widths (13 for the reference's models, else 16).
// part: [gridDim.x * 8][2 * 256 + 32] per-thread-slice partials (dW1 16x16, dW2 16x16, db1 16, db2 16).
template <int FP>
__global__ void __launch_bounds__(kGbwThreads, 1)
    gcn_bwd_kernel(const float* __restrict__ X, const float* __restrict__ dU, const float* __restrict__ adj,
                   const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2,
                   const float* __restrict__ b2, float* __restrict__ part, long long R, int S, int Fi, int Fh,
                   int Fo, int RB, int ldu) {
    constexpr int FPP = (FP + 1) / 2;
    extern __shared__ __align__(16) float smem[];
    const int NSG = ceil_div(S, kGbwSG);
    const int tid = threadIdx.x;
    const int astride = NSG * kGbwSG;   // table floats per row of the adjacency tables (one LDS.128 per group)
    const int SR = gcn_bwd_row_stride(S);   // padded slab row stride

    float* adjT = smem;
    float* adjN = adjT + (size_t)S * NSG * 8;
    float* w1d = adjN + (size_t)S * NSG * 8;
    float* w2d = w1d + kGbwW * kGbwW;
    float* w2t = w2d + kGbwW * kGbwW;
    float* b1s = w2t + kGbwW * kGbwW;
    float* b2s = b1s + kGbwW;
    float* s0 = b2s + kGbwW;                  // X (dense, on arrival) -> AX (padded)
    float* s1 = s0 + (size_t)RB * SR;          // G1 -> AG -> dZ1
    float* s2 = s1 + (size_t)RB * SR;          // dZ2 -> dAG
    float* sd = s2 + (size_t)RB * SR;          // dU (dense)
    uint64_t* bar = reinterpret_cast<uint64_t*>(sd + round_up(RB * ldu, 4));

    for (int e = tid; e < S * NSG * kGbwSG; e += kGbwThreads) {
        const int sp = e / (NSG * kGbwSG);
        const int c = e % (NSG * kGbwSG);
        const int qq = c / kGbwSG, i = c % kGbwSG;
        const int s = qq + NSG * i;       // thread qq owns stations qq, qq + NSG, ... (lanes = consecutive stations)
        const bool ok = s < S;
        adjT[e] = ok ? adj[(size_t)s * S + sp] : 0.0f;
        adjN[e] = ok ? adj[(size_t)sp * S + s] : 0.0f;
    }
    for (int e = tid; e < kGbwW * kGbwW; e += kGbwThreads) {
        const int f = e / kGbwW, fo = e % kGbwW;
        w1d[e] = (f < Fi && fo < Fh) ? W1[f * Fh + fo] : 0.0f;
        w2d[e] = (f < Fh && fo < Fo) ? W2[f * Fo + fo] : 0.0f;
        w2t[e] = (f < Fo && fo < Fh) ? W2[fo * Fo + f] : 0.0f;   // w2t[fo'][f'] = W2[f'][fo']
    }
    for (int e = tid; e < kGbwW; e += kGbwThreads) {
        b1s[e] = e < Fh ? b1[e] : 0.0f;
        b2s[e] = e < Fo ? b2[e] : 0.0f;
    }
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    __syncthreads();

    const int row_local = tid / NSG;
    const int q = tid % NSG;
    const long long nblocks = (R + RB - 1) / RB;
    const int in_cols = S * Fi, du_cols = ldu;   // dU rows are ldu floats apart (the GEMM that wrote them pads to 4)
    unsigned phase = 0;

    // reduction-phase coordinates: output tile (fi, fj) of 4 x 4, slice ks of the (row, station) index
    const int fi = (tid >> 2) & 3, fj = tid & 3, ks = tid >> 4;
    float2 aw1[4][2], aw2[4][2];
    float4 ab1 = make_float4(0.f, 0.f, 0.f, 0.f), ab2 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 4; ++i) aw1[i][0] = aw1[i][1] = aw2[i][0] = aw2[i][1] = make_float2(0.0f, 0.0f);

    // sum over the block's (row, station) pairs: this thread takes stations ks, ks + 8, ... of every row
    auto reduce = [&](const float* __restrict__ sa, const float* __restrict__ sb, int nrows_, float2 (&aw)[4][2],
                      float4& ab) {
        for (int row = 0; row < nrows_; ++row) {
            const float* pa = sa + (size_t)row * SR + fi * 4;
            const float* pb = sb + (size_t)row * SR + fj * 4;
#pragma unroll 2
            for (int k = ks; k < S; k += kGbwThreads / 16) {
                const float4 a = *reinterpret_cast<const float4*>(pa + k * kGbwFS);
                const float4 b = *reinterpret_cast<const float4*>(pb + k * kGbwFS);
                const float2 blo = make_float2(b.x, b.y), bhi = make_float2(b.z, b.w);
                aw[0][0] = __ffma2_rn(make_float2(a.x, a.x), blo, aw[0][0]);
                aw[0][1] = __ffma2_rn(make_float2(a.x, a.x), bhi, aw[0][1]);
                aw[1][0] = __ffma2_rn(make_float2(a.y, a.y), blo, aw[1][0]);
                aw[1][1] = __ffma2_rn(make_float2(a.y, a.y), bhi, aw[1][1]);
                aw[2][0] = __ffma2_rn(make_float2(a.z, a.z), blo, aw[2][0]);
                aw[2][1] = __ffma2_rn(make_float2(a.z, a.z), bhi, aw[2][1]);
                aw[3][0] = __ffma2_rn(make_float2(a.w, a.w), blo, aw[3][0]);
                aw[3][1] = __ffma2_rn(make_float2(a.w, a.w), bhi, aw[3][1]);
                if (fi == 0) { ab.x += b.x; ab.y += b.y; ab.z += b.z; ab.w += b.w; }
            }
        }
    };

    for (long long rb = blockIdx.x; rb < nblocks; rb += gridDim.x) {
        const long long r0 = rb * RB;
        const int nrows = (int)((R - r0) < RB ? (R - r0) : RB);
        const float* xsrc = X + (size_t)r0 * in_cols;
        const float* dsrc = dU + (size_t)r0 * du_cols;
        const size_t xbytes = (size_t)nrows * in_cols * 4, dbytes = (size_t)nrows * du_cols * 4;
        const bool bulk = ((reinterpret_cast<uintptr_t>(xsrc) | reinterpret_cast<uintptr_t>(dsrc)) & 15) == 0 &&
                          ((xbytes | dbytes) & 15) == 0;
        if (bulk) {
            if (tid == 0) {
                mbar_expect_tx(bar, (unsigned)(xbytes + dbytes));
                bulk_g2s(s0, xsrc, (unsigned)xbytes, bar);
                bulk_g2s(sd, dsrc, (unsigned)dbytes, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1;
        } else {
            for (int e = tid; e < nrows * in_cols; e += kGbwThreads) s0[e] = __ldg(xsrc + e);
            for (int e = tid; e < nrows * du_cols; e += kGbwThreads) sd[e] = __ldg(dsrc + e);
            __syncthreads();
        }
        const bool active = row_local < nrows && tid < RB * NSG;
        unsigned mask1[kGbwSG];
        float2 acc[kGbwSG][FPP];

        // ---- P1: AX = A.X (own stations) ; G1 = relu(AX.W1 + b1) ----
        if (active)
            gcn_bwd_agg<FPP, false>(acc, s0 + (size_t)row_local * in_cols, Fi, Fi, adjT + q * kGbwSG, astride, S);
        __syncthreads();   // every read of the dense X block is done: s0 becomes the padded AX slab
        if (active) {
#pragma unroll
            for (int i = 0; i < kGbwSG; ++i) {
                mask1[i] = 0u;
                const int s = q + NSG * i;
                if (s < S) {
                    float* ax = s0 + (size_t)row_local * SR + s * kGbwFS;
#pragma unroll
                    for (int fp = 0; fp < 8; ++fp)
                        *reinterpret_cast<float2*>(ax + 2 * fp) = fp < FPP ? acc[i][fp] : make_float2(0.0f, 0.0f);
                }
            }
#pragma unroll 1
            for (int fo0 = 0; fo0 < kGbwW; fo0 += 4) {
                float2 o[kGbwSG][2];
                gcn_bwd_xform4<FPP>(o, acc, w1d, fo0);
                const float4 bb = *reinterpret_cast<const float4*>(b1s + fo0);
#pragma unroll
                for (int i = 0; i < kGbwSG; ++i) {
                    const int s = q + NSG * i;
                    if (s < S) {
                        float4 g;
                        g.x = o[i][0].x + bb.x; g.y = o[i][0].y + bb.y; g.z = o[i][1].x + bb.z; g.w = o[i][1].y + bb.w;
                        g.x = g.x > 0.0f ? g.x : 0.0f; g.y = g.y > 0.0f ? g.y : 0.0f;
                        g.z = g.z > 0.0f ? g.z : 0.0f; g.w = g.w > 0.0f ? g.w : 0.0f;
                        mask1[i] |= ((g.x > 0.0f ? 1u : 0u) | (g.y > 0.0f ? 2u : 0u) | (g.z > 0.0f ? 4u : 0u) |
                                     (g.w > 0.0f ? 8u : 0u)) << fo0;
                        *reinterpret_cast<float4*>(s1 + (size_t)row_local * SR + s * kGbwFS + fo0) = g;
                    }
                }
            }
        }
        __syncthreads();

        // ---- P2: AG = A.G1 ; dZ2 = dU * [AG.W2 + b2 > 0] ----
        if (active)
            gcn_bwd_agg<FPP, true>(acc, s1 + (size_t)row_local * SR, kGbwFS, 2 * FPP, adjT + q * kGbwSG, astride, S);
        __syncthreads();   // every read of G1 is done: s1 becomes AG
        if (active) {
#pragma unroll
            for (int i = 0; i < kGbwSG; ++i) {
                const int s = q + NSG * i;
                if (s < S) {
                    float* ag = s1 + (size_t)row_local * SR + s * kGbwFS;
#pragma unroll
                    for (int fp = 0; fp < 8; ++fp)
                        *reinterpret_cast<float2*>(ag + 2 * fp) = fp < FPP ? acc[i][fp] : make_float2(0.0f, 0.0f);
                }
            }
#pragma unroll 1
            for (int fo0 = 0; fo0 < kGbwW; fo0 += 4) {
                float2 o[kGbwSG][2];
                gcn_bwd_xform4<FPP>(o, acc, w2d, fo0);
                const float4 bb = *reinterpret_cast<const float4*>(b2s + fo0);
#pragma unroll
                for (int i = 0; i < kGbwSG; ++i) {
                    const int s = q + NSG * i;
                    if (s < S) {
                        const float* du = sd + (size_t)row_local * du_cols + s * Fo + fo0;
                        float4 d;
                        d.x = (fo0 + 0 < Fo && o[i][0].x + bb.x > 0.0f) ? du[0] : 0.0f;
                        d.y = (fo0 + 1 < Fo && o[i][0].y + bb.y > 0.0f) ? du[1] : 0.0f;
                        d.z = (fo0 + 2 < Fo && o[i][1].x + bb.z > 0.0f) ? du[2] : 0.0f;
                        d.w = (fo0 + 3 < Fo && o[i][1].y + bb.w > 0.0f) ? du[3] : 0.0f;
                        *reinterpret_cast<float4*>(s2 + (size_t)row_local * SR + s * kGbwFS + fo0) = d;
                    }
                }
            }
        }
        __syncthreads();

        // ---- P3: dW2 += AG^T dZ2, db2 += colsum(dZ2) ; then dAG = dZ2 . W2^T in place ----
        reduce(s1, s2, nrows, aw2, ab2);
        if (active) {   // own dZ2 rows into registers (reads only) before anyone overwrites s2
#pragma unroll
            for (int i = 0; i < kGbwSG; ++i) {
                const int s = q + NSG * i;
                const float* dz = s2 + (size_t)row_local * SR + (s < S ? s : 0) * kGbwFS;
#pragma unroll
                for (int fp = 0; fp < FPP; ++fp) acc[i][fp] = *reinterpret_cast<const float2*>(dz + 2 * fp);
            }
        }
        __syncthreads();   // the reduction has read every dZ2
        if (active) {
#pragma unroll 1
            for (int fo0 = 0; fo0 < kGbwW; fo0 += 4) {
                float2 o[kGbwSG][2];
                gcn_bwd_xform4<FPP>(o, acc, w2t, fo0);
#pragma unroll
                for (int i = 0; i < kGbwSG; ++i) {
                    const int s = q + NSG * i;
                    if (s < S)
                        *reinterpret_cast<float4*>(s2 + (size_t)row_local * SR + s * kGbwFS + fo0) =
                            make_float4(o[i][0].x, o[i][0].y, o[i][1].x, o[i][1].y);
                }
            }
        }
        __syncthreads();

        // ---- P4: dG1 = A^T dAG ; dZ1 = dG1 * [G1 > 0] -> s1 ----
        if (active) {
            gcn_bwd_agg<FPP, true>(acc, s2 + (size_t)row_local * SR, kGbwFS, 2 * FPP, adjN + q * kGbwSG, astride, S);
#pragma unroll
            for (int i = 0; i < kGbwSG; ++i) {
                const int s = q + NSG * i;
                if (s < S) {
                    float* dz = s1 + (size_t)row_local * SR + s * kGbwFS;
#pragma unroll
                    for (int fp = 0; fp < 8; ++fp) {
                        float2 v = make_float2(0.0f, 0.0f);
                        if (fp < FPP) {
                            v.x = ((mask1[i] >> (2 * fp)) & 1u) ? acc[i][fp].x : 0.0f;
                            v.y = ((mask1[i] >> (2 * fp + 1)) & 1u) ? acc[i][fp].y : 0.0f;
                        }
                        *reinterpret_cast<float2*>(dz + 2 * fp) = v;
                    }
                }
            }
        }
        __syncthreads();

        // ---- P5: dW1 += AX^T dZ1, db1 += colsum(dZ1) ----
        reduce(s0, s1, nrows, aw1, ab1);
        __syncthreads();   // the slabs are free for the next block's bulk copies
    }

    // ---- per-thread partials: part[(cta * 8 + ks)][...] ----
    float* pp = part + ((size_t)blockIdx.x * (kGbwThreads / 16) + ks) * (2 * 256 + 32);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int f = fi * 4 + i;
        *reinterpret_cast<float4*>(pp + f * 16 + fj * 4) = make_float4(aw1[i][0].x, aw1[i][0].y, aw1[i][1].x, aw1[i][1].y);
        *reinterpret_cast<float4*>(pp + 256 + f * 16 + fj * 4) =
            make_float4(aw2[i][0].x, aw2[i][0].y, aw2[i][1].x, aw2[i][1].y);
    }
    if (fi == 0) {
        *reinterpret_cast<float4*>(pp + 512 + fj * 4) = ab1;
        *reinterpret_cast<float4*>(pp + 528 + fj * 4) = ab2;
    }
}

// dW1 [Fi][Fh], db1 [Fh], dW2 [Fh][Fo], db2 [Fo] = sums of the partials in a fixed order: one warp per output
// element, lane l adds partials l, l + 32, ... ascending, then a shuffle tree (deterministic; the serial loop
// over the 148 x 16 partials of round 1 took 0.10 ms).  grid = ceil(544 / 8) blocks of 256 threads.
__global__ void __launch_bounds__(256) gcn_bwd_finish_kernel(const float* __restrict__ part, int nparts, int Fi, int Fh,
                                                              int Fo, float* __restrict__ dW1, float* __restrict__ db1,
                                                              float* __restrict__ dW2, float* __restrict__ db2) {
    const int e = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (e >= 2 * 256 + 32) return;
    float s = 0.0f;
    for (int z = lane; z < nparts; z += 32) s += part[(size_t)z * (2 * 256 + 32) + e];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane != 0) return;
    if (e < 256) {
        const int f = e >> 4, fo = e & 15;
        if (f < Fi && fo < Fh) dW1[f * Fh + fo] = s;
    } else if (e < 512) {
        const int f = (e - 256) >> 4, fo = e & 15;
        if (f < Fh && fo < Fo) dW2[f * Fo + fo] = s;
    } else if (e < 528) {
        if (e - 512 < Fh) db1[e - 512] = s;
    } else {
        if (e - 528 < Fo) db2[e - 528] = s;
    }
}

}  // namespace wg
